#!/usr/bin/env python
"""bench.py -- pod x throttle admission checks/sec of the batched throttle-admission pass.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2] [--l2 rotate|flush] [--dump-outputs DIR]
  (N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" is ONE pass of the hot path over one synthetic snapshot: reconcile every throttle against the
running pods, (all-reduce the per-throttle partials when N>1), check every pending pod against every
throttle.  Workload at N=1 = BASELINE.json configs[1] (C2: 1k Throttles x 100k running x 10k pending, R=4).
N>1 is WEAK scaling: every rank holds a C2-sized row shard (its own 100k running + 10k pending rows) and a
replica of the same 1k throttles (thresholds scaled by N), i.e. one N-times-larger snapshot row-sharded
across the GPUs; `value` counts the checks of all ranks.  Beside the headline the line carries `configs`:
the other BASELINE shapes on this many GPUs (N=1: C2 with arrival-order rows, C3, C4, C5 on one device;
N>1: the shape BASELINE.json quotes for that N -- C3@2, C4@4, C5@8 -- STRONG-sharded by rows).

Timing (`--l2 rotate`, the default): E engine contexts hold E copies of the snapshot (E x footprint >= 2 x the
126 MB L2), the timed region launches K passes back to back cycling through them -- every pass reads inputs that
left L2 E-1 passes ago -- between ONE pair of CUDA events on the launching stream; ms_per_step = region / K.
`--l2 flush`: one context, a 512 MiB write + 512 MiB read between steps (outside the per-step event pairs).

One JSON line on rank 0 (keys per the driver contract + roofline + cpu_baseline).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pod_x_throttle_admission_checks_per_sec"
UNIT = "checks/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rows-scale", type=int, default=1,
                    help="NOT the headline: multiply the running/pending row counts of the config (steady-state efficiency probe)")
    ap.add_argument("--l2", default="rotate", choices=["rotate", "flush"],
                    help="how every timed pass gets cold inputs: rotate through enough snapshot copies to exceed L2 twice over (back-to-back "
                         "launches, one event pair) or flush L2 between steps (512 MiB write + 512 MiB read, per-step event pairs)")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only: skip the `configs` array")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (the pass result a caller receives) to DIR/<name>.npy "
                         "as float64, under 64 MB in all; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT = 60_000_000  # bytes of array data per dump: with the .npy headers, under 64 MB
THROTTLE_FIELDS = ("used", "used_present", "used_cnt", "throttled", "calc_thr", "calc_present", "calc_cnt", "override_active")
POD_FIELDS = {"running": ("run_bitmap",), "pending": ("pend_bitmap", "codes", "admit")}


def dump_outputs(out_dir, res):
    """Write a PassResult as float64 .npy files, one per field.  The per-throttle columns are written whole.  The per-pod arrays
    are written whole when everything fits in DUMP_LIMIT bytes; otherwise every array of one pod kind keeps the same seeded
    sample of rows, and the row numbers go to running_rows.npy / pending_rows.npy.  Bitmap and code words are 32-bit, so
    float64 holds them exactly; so does it hold the int64 sums below 2^53."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {f: getattr(res, f) for f in THROTTLE_FIELDS}
    fixed = 8 * sum(a.size for a in arrays.values())
    rows = {kind: getattr(res, fields[0]).shape[0] for kind, fields in POD_FIELDS.items()}
    row_bytes = {kind: 8 * sum(getattr(res, f)[:1].size for f in fields) for kind, fields in POD_FIELDS.items()}
    whole = sum(rows[k] * row_bytes[k] for k in POD_FIELDS)
    if fixed + whole <= DUMP_LIMIT:
        for fields in POD_FIELDS.values():
            arrays.update({f: getattr(res, f) for f in fields})
    else:
        frac = (DUMP_LIMIT - fixed) / sum(rows[k] * (row_bytes[k] + 8) for k in POD_FIELDS)  # + 8: the row number itself
        rng = np.random.default_rng(0)
        for kind, fields in POD_FIELDS.items():
            pick = np.sort(rng.choice(rows[kind], int(rows[kind] * frac), replace=False))
            arrays[kind + "_rows"] = pick
            arrays.update({f: getattr(res, f)[pick] for f in fields})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def measured_peaks():
    """HBM copy bandwidth measured on this pool's B200s by the driver; fallback per B200_PROFILING.md."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        for k in ("hbm_gbs", "hbm_gb_s", "hbm_GBps"):
            if k in d:
                return float(d[k]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_snapshot(config: str, rank: int, world: int, rows_scale: int = 1):
    from kube_throttler_b200 import synth

    if rows_scale > 1:
        base = synth.CONFIGS[config]
        snap = synth.generate(config, n=base["n"] * rows_scale, p=base["p"] * rows_scale, calibrate=False)
        snap.thr = snap.thr * rows_scale
        snap.thr_cnt = snap.thr_cnt * rows_scale
        return snap.normalize()
    snap = synth.generate(config)
    if world > 1:
        # weak scaling: same throttles on every rank, rank-specific pod rows, thresholds scaled with the snapshot
        own = synth.generate(config, seed=synth.CONFIGS[config]["seed"] + 1000 * (rank + 1), calibrate=False)
        snap.running, snap.pending = own.running, own.pending
        snap.thr = snap.thr * world
        snap.thr_cnt = snap.thr_cnt * world
        snap.normalize()
    return snap


def moved_bytes_estimate(snap, Wp):
    """What the pass HAS to move in this implementation (an estimate, for the honest reading of the roofline): the resident pod
    columns as stored (u32 row offsets instead of int64 labels, word info), the match / code words of each row's own namespace
    list (the bitmaps are maintained word by word, zero words are never rewritten), per-throttle tables and sums."""
    L, R, M = snap.L, snap.R, snap.m
    n, p = snap.running.n, snap.pending.n
    Lpad = (L + 7) // 8 * 8
    row = 4 * Lpad + 8 * R + 16
    words = 2  # words of a namespace's list, typical for namespaced Throttles
    return (n + p) * row + (n + p) * words * 4 + p * (words * 8 + 1) + p * (8 * R + 12) + M * (16 * R + 48 + 8 * (2 * R + 1) * 2)


def measured_traffic(config, rows_scale):
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_pass launch from THIS round's `ncu --set full` capture, if the
    committed summary (profiles/r2_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep) is for this workload."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        e = d.get(f"{config}x{rows_scale}")
        if e:
            pipes = {k: e[k] for k in ("sm_throughput_pct", "issue_active_pct", "alu_pipe_pct", "lsu_pipe_pct", "dram_throughput_pct") if k in e and e[k] == e[k]}
            return e["dram_bytes_read"] + e["dram_bytes_write"], e.get("source"), pipes
    except Exception:
        pass
    return None, None, None


def algorithmic_bytes(snap, Wp):
    """SURVEY.md section 8(d): bytes one pass must move, per kernel."""
    L, R, M = snap.L, snap.R, snap.m
    n, p = snap.running.n, snap.pending.n
    pod_row = 8 * L + 8 * R + 12
    s_thr = 16 * 2 + 8 * (2 * R + 2) + 16
    rec = n * pod_row + n * M / 8 + M * (2 * R + 1) * 8
    chk = p * pod_row + p * M / 8 + p * M / 4 + p + M * (16 + 16 * R)
    fin = M * s_thr + 2 * M * (2 * R + 2) * 8
    return dict(reconcile=rec, check=chk, finalize=fin, total=rec + chk + fin)


def workload_label(name, snap, world=1, sharded=None):
    rows = f"{snap.running.n} running x {snap.pending.n} pending" + (" per GPU" if world > 1 and not sharded else "")
    return f"{name}: {snap.m} throttles x {rows}, R={snap.R}, L={snap.L}"


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm for this path.  The reference is pure Go and no Go
    toolchain exists in this image (SURVEY.md 8c), so this times the ORACLE's reference-shaped port
    (oracle/ko_model.h: string maps, per-call selector construction, ResourceAmountOfPod recomputed per use)
    with every host thread (each worker pinned to its own CPU), on the same config.  Each step = one full pass over
    the snapshot (~0.1 s at C2 on 128 threads), K steps after W warm-ups as asked; `value` is taken from the MEDIAN
    step (thread start-up and allocator noise make single passes scatter)."""
    if rank != 0:
        return
    from oracle import ko

    snap = make_snapshot(args.config, 0, 1)
    threads = ko.hardware_threads()
    steps, warm = max(1, args.steps), max(0, args.warmup)
    times = []
    for i in range(warm + steps):
        res, tm = ko.object_evaluate(snap, threads=threads)
        if i >= warm:
            times.append(tm["total_s"])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    med = statistics.median(times)
    checks = snap.pending.n * snap.m
    value = checks / med
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * med, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": workload_label(args.config, snap), "timing": f"median of {steps} full passes (mean {1e3 * sum(times) / steps:.1f} ms, "
                                                                            f"min {1e3 * min(times):.1f}, max {1e3 * max(times):.1f})"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "full snapshot per step (reconcile of every throttle + PreFilter of every pending pod), workers pinned one per CPU"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "C++ restatement of the reference algorithm (not Go): no Go toolchain in this image",
    }
    print(json.dumps(line))


def gpu_local_cpus(dev_index):
    """The CPUs that sit next to the GPU (sysfs local_cpulist of the PCI function), or None."""
    try:
        import torch

        pr = torch.cuda.get_device_properties(dev_index)
        path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            if not part:
                continue
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return cpus or None
    except Exception:  # noqa: BLE001 -- diagnostics only
        return None


class Bench:
    """One rank's device, stream, rendezvous and L2-defeating buffers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
        torch.cuda.set_device(self.local_rank)
        self.all_cpus = os.sched_getaffinity(0)
        # pinned buffers are placed on the NUMA node of the allocating thread: keep this process next to its GPU, as a
        # deployment would (the CPU baseline below undoes it: its workers want every core)
        local = gpu_local_cpus(self.local_rank)
        self.host_affinity = "unchanged"
        if local:
            os.sched_setaffinity(0, local)
            self.host_affinity = f"{len(local)} GPU-local cpus"
        self.saved_stdout = None
        if self.world > 1:
            # NCCL prints its version banner on stdout at communicator creation; stdout belongs to the ONE JSON line of
            # rank 0, so file descriptor 1 points at stderr until the communicators exist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            sys.stdout.flush()
            self.saved_stdout = os.dup(1)
            os.dup2(2, 1)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.stream = torch.cuda.Stream()
        self.flush = self.drain = None
        self.align_t = torch.zeros(1, device="cuda")

    def restore_stdout(self):
        if self.saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(self.saved_stdout, 1)
            os.close(self.saved_stdout)
            self.saved_stdout = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def make_engines(self, snap, count):
        """`count` contexts on this rank's stream, each with its own copy of the snapshot (and, with several ranks, its own
        communicator + exchange windows: kt_comm_init is collective, every rank creates the same number in the same order)."""
        import kube_throttler_b200 as kt

        engines = []
        for _ in range(count):
            eng = kt.Engine(snap.R, snap.L, snap.LN, device=self.local_rank)
            eng.set_stream(self.stream.cuda_stream)
            if self.world > 1:
                uid = [kt.Engine.comm_unique_id() if self.rank == 0 else None]
                self.dist.broadcast_object_list(uid, src=0)
                eng.comm_init(uid[0], self.world, self.rank)
            eng.upload_snapshot(snap)
            engines.append(eng)
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()
        return engines

    def l2_flush(self):
        torch = self.torch
        if self.flush is None:
            self.flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
            self.drain = torch.empty(512 << 20, dtype=torch.uint8, device="cuda").view(torch.int64)
        self.flush.zero_()  # WRITE a buffer larger than L2: evicts the snapshot, every pass reads its inputs from HBM ...
        self.drain.sum()    # ... then READ another one, so that what sits in L2 is clean (no foreign write-backs inside the timed region)

    def time_passes(self, engines, now, steps, warmup, mode):
        """Device time of `steps` passes, max over ranks: (total ms, [per-step ms] or None)."""
        torch = self.torch
        E = len(engines)
        with torch.cuda.stream(self.stream):
            for i in range(max(warmup, 3, E)):
                if mode == "flush":
                    self.l2_flush()
                engines[i % E].evaluate(now)
        torch.cuda.synchronize()
        self.barrier()
        if mode == "rotate":
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(self.stream):
                # the host queues launches more slowly than a small pass runs: park the stream behind a spin kernel so that
                # all K launches are queued before the first one starts, and the device runs them back to back
                torch.cuda._sleep(int(steps * 60e3) + 2_000_000)
                if self.world > 1:
                    self.dist.all_reduce(self.align_t)  # line the ranks up (outside the events)
                a.record(self.stream)
                for i in range(steps):
                    engines[i % E].evaluate(now)
                b.record(self.stream)
            torch.cuda.synchronize()
            self.barrier()
            return self.max_over_ranks(a.elapsed_time(b)), None
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        with torch.cuda.stream(self.stream):
            for i, (a, b) in enumerate(evs):
                self.l2_flush()
                if self.world > 1:
                    # line the ranks up AFTER the flush and OUTSIDE the timed events: the flush kernels of different GPUs
                    # finish several microseconds apart, and a rank that enters the pass early would otherwise spend that
                    # skew waiting inside the pass's own exchange and book it as pass time
                    self.dist.all_reduce(self.align_t)
                a.record(self.stream)
                engines[i % E].evaluate(now)
                b.record(self.stream)
        torch.cuda.synchronize()
        self.barrier()
        step_ms = [a.elapsed_time(b) for a, b in evs]
        return self.max_over_ranks(sum(step_ms)), step_ms


def rotation_count(footprint_bytes, world):
    """Contexts whose snapshots together exceed twice the 126 MB L2 (an LRU-ish cache has then forgotten a snapshot by the
    time its turn comes again); capped -- with several ranks every context also carries a communicator."""
    need = int(np.ceil(2 * 126e6 / max(footprint_bytes, 1)))
    return max(1, min(need, 16 if world == 1 else 10))


def measure_config(bench, name, snap, steps, warmup, mode, peak, sharded=None, keep_engines=False):
    """Device-resident pass rate of one workload on this rank's GPU (all ranks' checks counted)."""
    from kube_throttler_b200 import abi  # noqa: F401

    probe = bench.make_engines(snap, 1)
    Wp = probe[0].words_per_row
    ab = algorithmic_bytes(snap, Wp)
    E = rotation_count(ab["total"], bench.world) if mode == "rotate" else 1
    engines = probe + (bench.make_engines(snap, E - 1) if E > 1 else [])
    total_ms, step_ms = bench.time_passes(engines, snap.now, steps, warmup, mode)
    launches = engines[0].timing().launches
    checks = snap.pending.n * snap.m * bench.world
    pass_ms = total_ms / steps
    achieved = ab["total"] / (pass_ms * 1e-3) / 1e9
    out = {
        "name": name, "workload": workload_label(name, snap, bench.world, sharded), "value": checks / (pass_ms * 1e-3), "unit": UNIT,
        "ms_per_step": pass_ms, "steps": steps, "launches_per_step": launches, "contexts_rotated": E,
        "roofline": {"bound": "hbm", "kernel": "k_pass", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "algorithmic_bytes": ab["total"], "frac_moved": moved_bytes_estimate(snap, Wp) / (pass_ms * 1e-3) / 1e9 / peak},
    }
    if sharded:
        out["parallelism"] = sharded
    if keep_engines:
        return out, engines, ab
    for e in engines:
        e.close()
    return out, None, ab


def measure_e2e(bench, eng, snap, Wp, args, checks_per_step):
    """The same metric end to end through the C ABI with HOST buffers: every step copies the packed pod rows host -> device
    (pinned memory), runs the pass and reads the results back (admit bits + non-zero check codes + per-throttle status)."""
    import kube_throttler_b200 as kt
    from kube_throttler_b200 import abi

    torch, world = bench.torch, bench.world
    r, p = snap.running, snap.pending
    pinned = []

    def pin(a, wc=False):
        b = kt.Pinned(a.shape, a.dtype, upload_only=wc)  # wc: write-combined, the CPU only writes these
        b.array[...] = a
        pinned.append(b)
        return b.array

    hr = abi.PodCols(pin(r.labels), pin(r.req), pin(r.present), pin(r.flags), pin(r.ns_id))
    hp = abi.PodCols(pin(p.labels), pin(p.req), pin(p.present), pin(p.flags), pin(p.ns_id))
    out = abi.PassResult.alloc(snap, Wp)
    codes_b, admit_b = kt.Pinned(out.codes.shape, np.uint32), kt.Pinned(out.admit.shape, np.uint8)
    h2d_wide = sum(a.nbytes for c in (hr, hp) for a in (c.labels, c.req, c.present, c.flags, c.ns_id))
    d2h_dense = codes_b.array.nbytes + admit_b.array.nbytes + sum(getattr(out, f).nbytes for f in
                                                                  ("used", "used_present", "used_cnt", "throttled", "calc_thr", "calc_present", "calc_cnt", "override_active"))
    # The snapshot crosses the host link in the packed transfer format when it is representable (kt_upload_pods_packed:
    # 16-bit label-pair indices, request columns as 1- or 2-byte dictionary codes, presence in the meta word; expanded to the
    # int64 HBM columns by a device kernel): the link, not the device, bounds an end-to-end pass.
    def pin_block(arrays, wc):
        """The device-bound columns of one pod kind carved out of ONE pinned block (16-byte aligned pieces): the library sees that
        they are contiguous and sends them across the link as one transfer."""
        offs, at = [], 0
        for a in arrays:
            offs.append(at)
            at += (a.nbytes + 15) & ~15
        blk = kt.Pinned((max(at, 16),), np.uint8, upload_only=wc)
        pinned.append(blk)
        views = []
        for a, o in zip(arrays, offs):
            v = blk.array[o:o + a.nbytes].view(a.dtype).reshape(a.shape)
            v[...] = a
            views.append(v)
        return views

    def packed_cols(wc):
        cols = []
        for pods in (r, p):
            try:
                c = abi.packed_pods(pods, code_requests=True)
                labels16, pairs, meta, req_codes, req_dict = pin_block([c.labels16, c.pairs, c.meta, c.req_codes, c.req_dict], wc)
                cols.append(abi.PackedPodCols(c.ns_bits, pairs, labels16, None, None, meta, req_dict, pin(c.req_dict_off), pin(c.req_code_bytes), req_codes))
            except ValueError:
                c = abi.packed_pods(pods)
                labels16, pairs, meta, req32 = pin_block([c.labels16, c.pairs, c.meta, c.req32], wc)
                cols.append(abi.PackedPodCols(c.ns_bits, pairs, labels16, req32, pin(c.req_shift), meta))
        return tuple(cols)

    try:
        packed, packed_wc = packed_cols(False), packed_cols(True)
    except ValueError:
        packed = packed_wc = None
    h2d = sum(c.nbytes for c in packed) if packed else h2d_wide

    sparse_cap = 4 * snap.pending.n + 1024
    ent_b = kt.Pinned((sparse_cap, 3), np.uint32)
    sparse_counts = []

    def fetch(e):
        # the check result comes back as admit[p] + the NON-ZERO code words (kt_get_check_sparse): what PreFilter needs of it;
        # a list that overflows falls back to the dense rows inside the timed step
        n = e.get_check_sparse(admit_b.array, ent_b.array)
        sparse_counts.append(n)
        if n > sparse_cap:
            e.get_check(codes_b.array, None)
        e.get_reconcile(out)

    def upload(e, cols):
        if cols:
            e.upload_pods_packed(abi.PODS_RUNNING, cols[0])
            e.upload_pods_packed(abi.PODS_PENDING, cols[1])
        else:
            e.upload_pods(abi.PODS_RUNNING, hr)
            e.upload_pods(abi.PODS_PENDING, hp)

    def step_wide():
        eng.upload_pods(abi.PODS_RUNNING, hr)
        eng.upload_pods(abi.PODS_PENDING, hp)
        eng.evaluate(snap.now)
        eng.get_check(codes_b.array, admit_b.array)
        eng.get_reconcile(out)

    src = [packed]

    def step():
        upload(eng, src[0])
        eng.evaluate(snap.now)
        fetch(eng)

    # ONE call per step (kt_step_submit: packed uploads + pass + result copies queued; kt_step_wait: one synchronisation); the
    # results land in the library's pinned block (status columns, admit bits, non-zero code words) and are read from there
    structs = {}

    def step_args(cols):
        key = id(cols)
        if key not in structs:
            structs[key] = [(c.n, c.struct()) for c in cols]  # the ctypes views of the pinned columns are built once
        return structs[key]

    import ctypes as C
    seen = []

    def consume(res):  # the caller looks at its result: the admit bits (a 10 KB read) and the count of rejected pairs
        sparse_counts.append(int(res.n_sparse))
        seen.append(C.cast(res.admit, C.POINTER(C.c_uint8))[0])

    def step_one_call():
        a_ = step_args(src[0])
        eng.step_submit(a_[0], a_[1], snap.now)
        consume(eng.step_wait())

    # what the host link of this box can do at all (one 64 MiB copy each way, from the same pinned allocator the step's buffers come
    # from -- a buffer pinned on the far NUMA node measures that node's link, not this step's): the floor of any e2e number
    probe_pin = kt.Pinned((64 << 20,), np.uint8)
    probe_pin.array[:] = 1
    probe_h, probe_d = torch.from_numpy(probe_pin.array), torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    link = {}
    for name, (dst, s_) in (("h2d", (probe_d, probe_h)), ("d2h", (probe_h, probe_d))):
        best = 0.0
        for _ in range(8):  # best of eight single copies, timed on the device: the first ones pay for the clock ramp
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            dst.copy_(s_, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            best = max(best, (64 << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        link[name + "_gbs"] = best
    del probe_h, probe_d, probe_pin

    def time_steps(fn, steps=None):
        steps = steps or args.e2e_steps
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        bench.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        bench.barrier()
        return checks_per_step * steps / bench.max_over_ranks(time.perf_counter() - t0)

    wide_value = time_steps(step_wide)
    eng.set_async_uploads(True)  # the pinned columns live for the whole run: no need to wait for each copy before queueing the next
    eng.set_sparse_check(sparse_cap)
    separate_calls_value = time_steps(step) if packed else None
    value = pinned_value = time_steps(step_one_call) if packed else time_steps(step)
    upload_memory = "pinned"
    if packed_wc:
        src[0] = packed_wc
        wc_value = time_steps(step_one_call)
        if wc_value > value:
            value, upload_memory = wc_value, "pinned write-combined"
        else:
            src[0] = packed
    serial_value = value
    # Double-buffered steps: a second context (own stream, own snapshot buffers) is handed the NEXT step while this step's
    # pass runs and its results come back -- H2D, the pass and D2H of consecutive steps overlap; every step still copies its
    # inputs in and its results out and is waited for.  Single GPU only (a second context would need a second peer window set).
    pipelined, depth_values, best_depth, host_us = None, {}, 0, {}
    if world == 1 and packed:
        # D contexts in a ring: step k+D-1 is submitted before step k is waited for.  One step's latency (two uploads, two unpack
        # launches, the pass, three result copies, all in stream order, plus the host's submit and wake-up) is ~2.5x the time its
        # bytes need on the link, so two contexts do not fill the link yet; three or four do.
        ring = [eng]
        try:
            a_ = step_args(src[0])
            for depth in (2, 4, 6, 8):
                while len(ring) < depth:
                    e2 = kt.Engine(snap.R, snap.L, snap.LN, device=bench.local_rank)
                    st2 = torch.cuda.Stream()
                    e2._bench_stream = st2  # keeps the stream alive as long as the engine
                    e2.set_stream(st2.cuda_stream)
                    e2.upload_snapshot(snap)
                    e2.set_async_uploads(True)
                    e2.set_sparse_check(sparse_cap)
                    ring.append(e2)
                turn = [0]
                for k in range(depth - 1):
                    ring[k].step_submit(a_[0], a_[1], snap.now)

                host_ns = [0, 0, 0]  # inside kt_step_submit, inside kt_step_wait, steps

                def step_pipelined():
                    t0_ = time.perf_counter_ns()
                    ring[(turn[0] + depth - 1) % depth].step_submit(a_[0], a_[1], snap.now)  # step k+D-1 is queued on its own stream ...
                    t1_ = time.perf_counter_ns()
                    consume(ring[turn[0] % depth].step_wait())                              # ... while step k finishes
                    host_ns[0] += t1_ - t0_
                    host_ns[1] += time.perf_counter_ns() - t1_
                    host_ns[2] += 1
                    turn[0] += 1

                v = time_steps(step_pipelined, 4 * args.e2e_steps)
                for k in range(depth - 1):
                    ring[(turn[0] + k) % depth].step_wait()
                depth_values[str(depth)] = v
                host_us[str(depth)] = {"submit": host_ns[0] / host_ns[2] / 1e3, "wait": host_ns[1] / host_ns[2] / 1e3}
                if pipelined is None or v > pipelined:
                    pipelined, best_depth = v, depth
        except Exception as e:  # noqa: BLE001 -- the serial number stands
            print(f"pipelined e2e unavailable: {e}", file=sys.stderr)
        for e2 in ring[1:]:
            try:
                e2.sync()
                e2.close()
            except Exception:  # noqa: BLE001
                pass
    if pipelined and pipelined > value:
        value = pipelined
    eng.set_sparse_check(0)
    eng.set_async_uploads(False)
    n_sparse = max(sparse_counts) if sparse_counts else 0
    # the fetch asks for the last count + 25 % + 256 entries
    d2h = d2h_dense - codes_b.array.nbytes + (12 * min(n_sparse + n_sparse // 4 + 256, sparse_cap) + 4 if n_sparse <= sparse_cap else 12 * sparse_cap + 4 + codes_b.array.nbytes)
    floor = checks_per_step / world / (h2d / (link["h2d_gbs"] * 1e9) + d2h / (link["d2h_gbs"] * 1e9)) * world
    return {"value": value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
            "path": (("kt_step_submit (kt_upload_pods_packed x2 + kt_evaluate + result copies) + kt_step_wait, pinned host buffers; " +
                      (f"{best_depth} contexts in a ring: step k+{best_depth - 1} is submitted before step k is waited for" if pipelined and value == pipelined else "one context, serial"))
                     if packed else "kt_upload_pods x2 + kt_evaluate + kt_get_check_sparse + kt_get_reconcile (pinned host buffers)"),
            "serial": {"value": serial_value, "note": "one context: submit, wait, submit, ..."},
            "double_buffered": {"value": pipelined, "contexts": best_depth, "by_contexts": depth_values, "host_us_per_step": host_us,
                                "note": "D contexts in a ring: the uploads of the next steps overlap this step's pass and download; every step still copies its inputs in and its results out and is waited for"},
            "separate_calls": {"value": separate_calls_value, "note": "kt_upload_pods_packed x2 + kt_evaluate + kt_get_check_sparse + kt_get_reconcile, one context"},
            "sparse_check_entries": n_sparse, "upload_memory": upload_memory, "pinned_upload_value": pinned_value, "host_affinity": bench.host_affinity,
            "wide_int64_upload": {"value": wide_value, "h2d_bytes_per_step": h2d_wide, "d2h_bytes_per_step": d2h_dense},
            "host_link_gbs": link, "link_floor_value": floor, "frac_of_link_floor": value / floor,
            "admit_fraction": float(admit_b.array.mean())}


def measure_plugin(device):
    """The reference-facing plugin surface (include/kt_host.h) on this device: see tools/plugin_bench.py."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import plugin_bench

    return plugin_bench.run(device)


def shard_snapshot(snap, rank, world):
    """STRONG scaling of a BASELINE shape: contiguous row ranges of the ONE snapshot (SURVEY.md 8e), throttles replicated."""
    from kube_throttler_b200 import shard

    return shard.shard_snapshot(snap, rank, world)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return
    bench = Bench(args)
    rank, world, local_rank = bench.rank, bench.world, bench.local_rank
    torch, dist = bench.torch, bench.dist
    if world != args.gpus and world > 1:
        args.gpus = world

    import kube_throttler_b200 as kt
    from kube_throttler_b200 import abi, synth

    peak, peak_src = measured_peaks()
    mode = args.l2
    snap = make_snapshot(args.config, rank, world, args.rows_scale)

    # ---- headline: device-resident timing, W warm-up passes, then exactly K timed ones ------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_wall0 = time.perf_counter()
    head, engines, ab = measure_config(bench, args.config, snap, args.steps, args.warmup, mode, peak, keep_engines=True)
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    bench.restore_stdout()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engines[(args.steps - 1) % len(engines)].download())  # the context of the last timed pass
    eng = engines[0]
    Wp = eng.words_per_row
    launches_per_step = head["launches_per_step"]
    checks_per_step = snap.pending.n * snap.m * world
    pass_ms = head["ms_per_step"]

    # the other way of keeping inputs cold, for comparison (same contexts, fewer steps)
    other_mode = "flush" if mode == "rotate" else "rotate"
    alt_ms, _ = bench.time_passes(engines if other_mode == "rotate" else engines[:1], snap.now, min(args.steps, 20), 3, other_mode)
    alt_ms /= min(args.steps, 20)

    # ---- per-kernel device times (library events; the three PDL-chained kernels), L2 flushed ---------
    eng.enable_timing(True)
    per = {"reconcile": [], "allreduce": [], "finalize": [], "check": []}
    for _ in range(min(args.steps, 20)):
        with torch.cuda.stream(bench.stream):
            bench.l2_flush()
            eng.evaluate(snap.now)
        torch.cuda.synchronize()
        t = eng.timing()
        per["reconcile"].append(t.reconcile_ms); per["allreduce"].append(t.allreduce_ms)
        per["finalize"].append(t.finalize_ms); per["check"].append(t.check_ms)
    eng.enable_timing(False)
    kernel_ms = {k: float(np.mean(v)) for k, v in per.items()}
    rec_gbs = ab["reconcile"] / (kernel_ms["reconcile"] * 1e-3) / 1e9
    # The timed region launches ONE kernel per step (k_pass: match + reconcile + finalize + decide tiles), so that is the
    # dominant kernel and its average launch duration is region / K.  The three-kernel breakdown (kt_enable_timing switches
    # the library to its PDL-chained launch path) is reported beside it: `reconcile` is where the bytes are.
    # traffic: dram__bytes_read.sum + dram__bytes_write.sum of one k_pass launch needs ncu, which bench.py does not run: they are
    # read from the committed capture of this workload (profiles/r2_traffic.json <- tools/ncu_traffic.py <- the .ncu-rep), with
    # the pipe utilisations of the same capture (SURVEY 8(d): ALU pipe next to HBM %); null when there is no capture.
    roofline = dict(head["roofline"])
    traffic, traffic_src, pipes = measured_traffic(args.config, args.rows_scale)
    moved = moved_bytes_estimate(snap, Wp)
    roofline.update({"traffic": traffic, "traffic_source": traffic_src or "none committed for this workload (ncu is not run inside bench.py)",
                     "pipes_under_ncu": pipes, "moved_bytes_estimate": moved, "frac_moved": moved / (pass_ms * 1e-3) / 1e9 / peak,
                     "note": "achieved / frac use SURVEY.md 8(d)'s algorithmic bytes (dense bitmap written once per pass); the pass maintains its "
                             "bitmaps word by word and stores int32 row offsets, so it moves fewer bytes than that -- frac_moved is the same time "
                             "against the bytes it has to move (latency-bound at this size either way)",
                     "peak_source": peak_src, "kernel_ms": pass_ms, "timing": mode,
                     "other_timing": {"mode": other_mode, "ms_per_step": alt_ms, "frac": ab["total"] / (alt_ms * 1e-3) / 1e9 / peak},
                     "chained_kernel_ms": kernel_ms,
                     "chained_reconcile": {"algorithmic_bytes": ab["reconcile"], "achieved": rec_gbs, "frac": rec_gbs / peak}})

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D pods, pass, D2H results ---------
    e2e = measure_e2e(bench, eng, snap, Wp, args, checks_per_step)
    for e in engines:
        e.close()

    # ---- the other BASELINE shapes ---------------------------------------------------------------------
    extras = []
    if not args.no_extras and args.rows_scale == 1 and args.config == "C2":
        k = max(3, min(args.steps, 10))
        if world == 1:
            # (C3-host-layout: C3 with its ClusterThrottles in the order the plugin surface lays its device columns out in -- by the
            # set of namespaces their namespaceSelectors admit, kt_host.cc reorder_columns: 8.9 words per pod instead of 15.3)
            plan = [("C2-unsorted", lambda: synth.generate("C2", sort_by_namespace=False)), ("C3", lambda: synth.generate("C3")),
                    ("C4", lambda: synth.generate("C4")), ("C5", lambda: synth.generate("C5")),
                    ("C3-host-layout", lambda: synth.generate("C3", column_layout=True))]
        else:
            cfg = {2: "C3", 4: "C4", 8: "C5"}.get(world)
            plan = [(f"{cfg}@{world}", lambda: shard_snapshot(synth.generate(cfg), rank, world))] if cfg else []
        for name, gen in plan:
            try:
                s2 = gen()
                res, _, _ = measure_config(bench, name, s2, k, 3, mode, peak, sharded=f"row-shard x{world} (strong)" if world > 1 else None)
                if world > 1:  # strong scaling: the checks of the ONE snapshot
                    res["value"] = bench.max_over_ranks(0.0) * 0 + sum_over_ranks(bench, s2.pending.n) * s2.m / (res["ms_per_step"] * 1e-3)
                extras.append(res)
                del s2
            except Exception as e:  # noqa: BLE001 -- an extra that fails must not take the headline with it
                extras.append({"name": name, "error": f"{type(e).__name__}: {e}"})

    # ---- plugin level: the reference-facing surface (include/kt_host.h) on this device ------------------
    plugin = None
    if rank == 0 and world == 1 and not args.no_extras and args.rows_scale == 1:
        try:
            plugin = measure_plugin(local_rank)
        except Exception as e:  # noqa: BLE001
            plugin = {"error": f"{type(e).__name__}: {e}"}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only): bounded, ~seconds ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.rows_scale == 1:
        from oracle import ko  # checker / baseline only -- never on the measured GPU path

        os.sched_setaffinity(0, bench.all_cpus)  # its workers pin themselves, one per CPU of the whole box
        threads = ko.hardware_threads()
        times = []
        for _ in range(6):
            _, tm = ko.object_evaluate(snap, threads=threads)
            times.append(tm)
        tm = sorted(times[1:], key=lambda x: x["total_s"])[len(times[1:]) // 2]
        cpu = {"value": snap.pending.n * snap.m / tm["total_s"], "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"median of 5 full {args.config} passes after 1 warm-up (reconcile {tm['reconcile_s']:.3f}s + check {tm['check_s']:.3f}s), "
                         "workers pinned one per CPU; C++ restatement of the reference algorithm (not Go)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": pass_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": workload_label(args.config, snap, world), "per_gpu_rows": [snap.running.n, snap.pending.n], "throttles": snap.m,
                       "l2": (f"inputs larger than L2: {head['contexts_rotated']} snapshot copies ({head['contexts_rotated'] * ab['total'] / 1e6:.0f} MB of pass "
                              "traffic) rotated, K passes back to back between one CUDA-event pair" if mode == "rotate" else
                              "flushed between steps, outside the timed events: 512 MiB memset then 512 MiB read (L2 holds clean foreign lines)"),
                       "parallelism": f"row-shard x{world}", "admit_fraction": e2e.pop("admit_fraction")},
            "e2e": e2e, "gpu_launches": launches_per_step * args.steps, "roofline": roofline, "configs": extras, "e2e_plugin": plugin,
            "cpu_baseline": cpu, "clocks": clocks, "wall_s_timed_region": t_wall,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def sum_over_ranks(bench, x):
    t = bench.torch.tensor([float(x)], dtype=bench.torch.float64, device="cuda")
    if bench.world > 1:
        bench.dist.all_reduce(t)
    return float(t.item())


if __name__ == "__main__":
    main()
