#!/usr/bin/env python
"""bench.py — Avro->Arrow direct-decode throughput on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload kafka|flat|wide] [--records R]
    python bench.py --impl reference ...        # the CPU arm: the oracle port on the usable host cores
    python bench.py --gpus N --gather ...        # C5: shards decoded per GPU, then gathered into single RecordBatches
    python bench.py --dump-outputs DIR ...       # also write the last timed step's output to DIR/*.npy (dump_outputs)

A "step" is one pass of the hot path over one batch of synthetic Avro records (C3: 10 M records, 8 output chunks):
  value     records/s with the packed input already resident in HBM and the Arrow buffers left in HBM
            (rv_decode_device); CUDA events on the launch stream; max over ranks.
  e2e       the same batch through the reference-facing C-ABI call rv_decode_host with HOST buffers:
            H2D of the packed input (pinned), the kernel, D2H of every Arrow buffer (pinned).
  roofline  algorithmic bytes (input + i64 offsets + every exported Arrow buffer) of the one fused decode kernel /
            its CUDA-event duration / measured HBM peak; path_frac = the same bytes / the whole device-resident step.
  cpu_baseline  the C oracle (row-at-a-time port of fast_decode.rs) on the usable host cores, the same 10 M records,
            with the reference's own num_chunks = 8 and with 4 chunks per core; medians.
  c1/c2/c4  the other BASELINE.json configurations (C1 through the Python surface, next to the README's 1.17 ms).
Multi-GPU: records shard by message with no data-path collective (weak scaling: R records per GPU).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "avro_to_arrow_records_per_sec"
UNIT = "records/s"
WORKLOAD_DESC = {
    "kafka": "C3: scripts/generate_avro.py Kafka schema (nullable unions, nested structs, array, map, 4-variant union, enum)",
    "flat": "C2: flat primitives (benches/common/mod.rs FLAT_PRIMITIVES)",
    "wide": "C4: four 8-variant sparse unions + three maps (divergence stress)",
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="kafka", choices=list(WORKLOAD_DESC))
    ap.add_argument("--records", type=int, default=10_000_000, help="records per GPU")
    ap.add_argument("--num-chunks", type=int, default=8, help="output batches per call (README bench: 8)")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--gather", action="store_true", help="C5: gather the shards' batches into single RecordBatches on rank 0")
    ap.add_argument("--no-extras", action="store_true", help="skip C1/C2/C4, encode and the CPU baseline (main line only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed device-resident step's output (a seeded sample of "
                    "its rows, every Arrow array flattened to float32/float64) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gather):
        ap.error("--dump-outputs applies to the GPU arm's main line (not --impl reference or --gather)")
    return args


def config_of(args, world):
    """Identical for the GPU arm and the reference arm (the driver compares them)."""
    return {"workload": WORKLOAD_DESC[args.workload], "records_per_gpu": args.records, "num_chunks": args.num_chunks, "seed": args.seed,
            "l2": "no flush: every step streams its whole input and output, an order of magnitude larger than the 126 MB L2",
            "sharding": "records by message, contiguous ranges per rank, no collective"}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def usable_cores():
    """Cores this process may really use: the affinity mask capped by the cgroup CPU quota (a box that shows 128
    CPUs under a 16-CPU quota runs 128 threads eight times slower than 16)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    quota = float(parts[0]) / float(parts[1])
            else:
                q = float(parts[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        quota = q / float(f2.read().split()[0])
            break
        except Exception:
            continue
    n = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return n, aff, quota


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed regions run."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.active = threading.Event()
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
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10}
        while not self._stop_evt.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    try:
                        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for k, bit in names.items():
                        if mask & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
            time.sleep(0.010)

    def stop(self):
        self._stop_evt.set()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's per_datum_deserialize_threaded
# ------------------------------------------------------------------------------------------------------
def cpu_arm(args, steps, warmup, emit_line, world=1):
    import workloads
    from oracle import pyoracle as po
    co = po.COracle()
    cores, aff, quota = usable_cores()
    co.lib.orc_set_pin(1)  # worker t -> the t-th allowed CPU: steadier on shared boxes
    n = args.records
    schema, data, offsets = workloads.generate(args.workload, n, seed=args.seed)
    # num_chunks is the reference's own tuning knob: its benches and README use 8 (ruhvro/benches/common/mod.rs:10);
    # four chunks per core keep every worker busy to the end and each chunk's builders cache-resident (the fastest
    # setting of this implementation).  Both are timed; the line's value is the better one.
    settings = [("k=%d (the reference's NUM_CHUNKS)" % args.num_chunks, args.num_chunks), ("k=4 x usable cores", 4 * cores)]
    results = []
    for label, k in settings:
        threads = max(1, min(cores, k))
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            co.decode_threaded_packed(schema, data, offsets, n, k, threads, materialize=False)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
        med = statistics.median(times)
        results.append({"setting": label, "num_chunks": k, "threads": threads, "records_per_s": n / med, "ms_per_step_median": 1000.0 * med,
                        "ms_per_step_min": 1000.0 * min(times), "ms_per_step_max": 1000.0 * max(times)})
    best = max(results, key=lambda r: r["records_per_s"])
    base = {"value": best["records_per_s"], "unit": UNIT, "cores": best["threads"], "kind": "port",
            "sample": f"all {n} records of the workload per pass, {len(times)} timed passes per setting, medians "
                      f"(oracle/avro_oracle.c, threads pinned; the Rust reference cannot be built here)",
            "settings": results, "cpus": {"usable": cores, "affinity": aff, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}}
    if emit_line:
        line = {"impl": "reference", "metric": METRIC, "value": best["records_per_s"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
                "warmup": warmup, "ms_per_step": best["ms_per_step_median"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config_of(args, world),
                "cpu_baseline": base,
                "e2e": {"value": best["records_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
    return base


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, args, rank, local_rank, world):
        import torch
        import pyruhvro_b200 as pr
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        self.torch, self.pr, self.L = torch, pr, pr.lib
        self.dev = torch.device("cuda", local_rank)
        self.stream = torch.cuda.current_stream()
        self.pinned_blocks = []

    def alloc_pinned(self, nbytes):
        p = self.L.rv_host_alloc(nbytes)
        if not p:
            raise SystemExit("rv_host_alloc failed: " + self.pr._last_error())
        self.pinned_blocks.append(p)
        return np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(p))

    def free_pinned(self):
        for p in self.pinned_blocks:
            self.L.rv_host_free(p)
        self.pinned_blocks = []

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier(device_ids=[self.local_rank])

    def max_over_ranks(self, v):
        if self.world == 1:
            return v
        import torch.distributed as dist
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def load(self, workload, n, seed, r0=0):
        import workloads
        torch = self.torch
        schema_json, h_data, h_off = workloads.generate(workload, n, seed=seed, r0=r0, alloc=self.alloc_pinned)
        total_in = int(h_off[n])
        d_data = torch.empty(total_in + 64, dtype=torch.uint8, device=self.dev)
        d_off = torch.empty(n + 1, dtype=torch.int64, device=self.dev)
        d_data[:total_in].copy_(torch.from_numpy(h_data))
        d_off.copy_(torch.from_numpy(h_off))
        torch.cuda.synchronize()
        return {"schema_json": schema_json, "schema": self.pr._get_or_parse_schema(schema_json), "h_data": h_data, "h_off": h_off,
                "d_data": d_data, "d_off": d_off, "n": n, "total_in": total_in}

    def step_device(self, w, k):
        h = ctypes.c_void_p()
        rc = self.L.rv_decode_device(w["schema"].handle, w["d_data"].data_ptr(), w["d_off"].data_ptr(), w["n"], k, self.stream.cuda_stream, ctypes.byref(h))
        if rc:
            raise SystemExit("rv_decode_device: " + self.pr._last_error())
        return h

    def step_host(self, w, k):
        h = ctypes.c_void_p()
        rc = self.L.rv_decode_host(w["schema"].handle, w["h_data"].ctypes.data, w["h_off"].ctypes.data, w["n"], k, ctypes.byref(h))
        if rc:
            raise SystemExit("rv_decode_host: " + self.pr._last_error())
        return h

    def time_device(self, w, k, steps, warmup, sampler=None, keep_last=False):
        """Device-resident decode: CUDA events around `steps` calls, max over ranks.  With keep_last the last step's
        result handle is returned as "last" instead of freed (the caller frees it)."""
        torch, L = self.torch, self.L
        last = None
        arrow_bytes = buffer_bytes = 0
        for _ in range(warmup):
            h = self.step_device(w, k)
            arrow_bytes, buffer_bytes = L.rv_result_arrow_bytes(h), L.rv_result_buffer_bytes(h)
            L.rv_result_free(h)
        kt = np.zeros(6, dtype=np.float64)
        tbuf = (ctypes.c_float * 6)()
        launches = passes = slow = 0
        self.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.active.set()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for i in range(steps):
            h = self.step_device(w, k)
            L.rv_last_timings(tbuf, 6)
            kt += np.frombuffer(tbuf, dtype=np.float32)
            launches += L.rv_last_launch_count()
            passes = max(passes, L.rv_last_passes())
            slow += L.rv_last_slow_tiles()
            if keep_last and i == steps - 1:
                last = h
            else:
                L.rv_result_free(h)
        e1.record(self.stream)
        torch.cuda.synchronize()
        if sampler:
            sampler.active.clear()
        self.barrier()
        ms_total = self.max_over_ranks(e0.elapsed_time(e1))
        return {"ms_per_step": ms_total / steps, "kernel_ms": kt / steps, "launches": launches, "passes": passes, "slow_tiles": slow,
                "arrow_bytes": arrow_bytes, "buffer_bytes": buffer_bytes, "last": last}

    def time_host(self, w, k, steps, warmup, sampler=None):
        """End to end through rv_decode_host (pinned host in, pinned host out), wall clock, max over ranks."""
        torch, L = self.torch, self.L
        buffer_bytes = 0
        for _ in range(warmup):
            h = self.step_host(w, k)
            buffer_bytes = L.rv_result_buffer_bytes(h)
            L.rv_result_free(h)
        tbuf = (ctypes.c_float * 6)()
        self.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.active.set()
        t0 = time.perf_counter()
        h2d_ms = d2h_ms = 0.0
        for _ in range(steps):
            h = self.step_host(w, k)
            L.rv_last_timings(tbuf, 6)
            h2d_ms += tbuf[4]
            d2h_ms += tbuf[5]
            L.rv_result_free(h)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        if sampler:
            sampler.active.clear()
        self.barrier()
        my_ms = 1000.0 * s / steps
        s = self.max_over_ranks(s)
        idx = 8 * (w["n"] + 1)
        h2d_b, d2h_b = w["total_in"] + idx, buffer_bytes
        per_rank = None
        if self.world > 1:  # every rank's own step time and copy-engine rates (NUMA placement shows up here)
            import torch.distributed as dist
            mine = self.torch.tensor([my_ms, h2d_b / max(h2d_ms / steps, 1e-9) / 1e6, d2h_b / max(d2h_ms / steps, 1e-9) / 1e6],
                                     dtype=self.torch.float64, device=self.dev)
            allv = [self.torch.zeros_like(mine) for _ in range(self.world)]
            dist.all_gather(allv, mine)
            per_rank = [{"rank": r, "ms_per_step": float(v[0]), "h2d_gbs_while_copying": float(v[1]), "d2h_gbs_while_copying": float(v[2])}
                        for r, v in enumerate(allv)]
        return {"ms_per_step": 1000.0 * s / steps, "h2d_bytes": h2d_b, "d2h_bytes": d2h_b, "per_rank": per_rank,
                # copy-engine time summed over the call's chunks (they overlap each other and the kernels)
                "h2d_busy_ms": h2d_ms / steps, "d2h_busy_ms": d2h_ms / steps,
                "h2d_gbs_while_copying": h2d_b / max(h2d_ms / steps, 1e-9) / 1e6, "d2h_gbs_while_copying": d2h_b / max(d2h_ms / steps, 1e-9) / 1e6}

    def roofline(self, w, dev, peak, peak_src):
        idx = 8 * (w["n"] + 1)
        algo = w["total_in"] + idx + dev["arrow_bytes"]
        kms = float(dev["kernel_ms"][0])
        gbs = algo / (kms * 1e-3) / 1e9 if kms > 0 else 0.0
        return {"bound": "hbm", "kernel": "rvj_fused" if self.pr.last_walker() == "jit" else "fused_kernel", "achieved": gbs, "peak": peak,
                "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes": algo, "kernel_ms": kms, "peak_source": peak_src,
                "path_frac": algo / (dev["ms_per_step"] * 1e-3) / 1e9 / peak, "path_ms": dev["ms_per_step"],
                "extra_pass_ms": float(dev["kernel_ms"][1]), "null_count_kernel_ms": float(dev["kernel_ms"][3]),
                "passes_per_step": dev["passes"], "walker": self.pr.last_walker(), "slow_tiles": dev["slow_tiles"]}


def traffic_of(workload, n):
    """DRAM bytes per launch of the fused kernel from the committed ncu capture (profiles/traffic.json, written from an
    `ncu --set full` run; the first entry for the workload and size is the current build's, older ones are kept marked
    `superseded`)."""
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(tpath) as f:
            tj = json.load(f)
        for e in tj.get("entries", []):
            if e.get("workload") == workload and e.get("records") == n and e.get("kernel") == "rvj_fused":
                return e.get("dram_bytes"), e.get("capture")
    except Exception:
        pass
    return None, None


def bind_to_gpu_node(torch, local_rank):
    """Runs this rank's threads on the CPUs of its GPU's NUMA node (what `numactl --cpunodebind` would do per rank): the
    calling thread's driver calls, the template / read-back copies and the library's workers stay on the GPU's socket.
    Returns the node, or None when it cannot be determined (then nothing changes)."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        cpus = set()
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def parity_check(b, w, k):
    """Outside every timed region: the exact arena the bench times, decoded through the host C ABI and through the
    device-resident path, compared buffer-for-buffer with the C oracle (the checker; never the thing measured)."""
    from oracle import pyoracle as po
    from tests.parity import assert_matches_oracle
    co = po.COracle()
    pr, L = b.pr, b.L
    got = pr.decode_packed(w["h_data"], w["h_off"], w["n"], w["schema_json"], k)
    assert_matches_oracle(co, got, w["schema_json"], w["h_data"], w["h_off"], w["n"], k, full_validate=False)
    del got
    h = b.step_device(w, k)
    pr._check(L.rv_result_to_host(h))
    assert_matches_oracle(co, pr._export_batches(h.value, w["schema"]), w["schema_json"], w["h_data"], w["h_off"], w["n"], k, full_validate=False)
    return True


DUMP_MAX_BYTES = 64 << 20
DUMP_MAX_ROWS = 1 << 15


def flatten_arrow(name, arr, out):
    """One Arrow array -> numpy float arrays in `out`, keyed by dotted path: validity (1/0), list and map lengths, union
    type ids, string and binary lengths and bytes, fixed-width values.  A 64-bit integer becomes a (high, low) pair of
    32-bit halves so that float64 holds it exactly."""
    import pyarrow as pa
    import pyarrow.compute as pc
    t, n = arr.type, len(arr)
    if not pa.types.is_union(t):          # a union has no validity of its own: its children carry it
        out[name + ".valid"] = arr.is_valid().to_numpy(zero_copy_only=False).astype(np.float32)
    if pa.types.is_struct(t):
        for i in range(t.num_fields):
            flatten_arrow(name + "." + t.field(i).name, arr.field(i), out)
    elif pa.types.is_list(t) or pa.types.is_large_list(t) or pa.types.is_map(t):
        off = arr.offsets.to_numpy().astype(np.int64)
        lens = np.diff(off)
        lens[~arr.is_valid().to_numpy(zero_copy_only=False)] = 0    # what a null list spans is not part of the value
        out[name + ".len"] = lens.astype(np.float32)
        ends = np.cumsum(lens)
        items = np.arange(int(ends[-1]) if n else 0) + np.repeat(off[:-1] - (ends - lens), lens)
        flatten_arrow(name + ".item", arr.values.take(pa.array(items, type=pa.int64())), out)
    elif pa.types.is_union(t):
        out[name + ".type_id"] = arr.type_codes.to_numpy().astype(np.float32)
        if t.mode == "dense":
            out[name + ".offset"] = arr.offsets.to_numpy().astype(np.float64)
        for i in range(t.num_fields):
            flatten_arrow(name + "." + t.field(i).name, arr.field(i), out)
    elif pa.types.is_dictionary(t):
        flatten_arrow(name + ".index", arr.indices, out)
        flatten_arrow(name + ".dictionary", arr.dictionary, out)
    elif pa.types.is_null(t):
        pass
    elif pa.types.is_boolean(t):
        out[name] = arr.fill_null(False).to_numpy(zero_copy_only=False).astype(np.float32)
    elif pa.types.is_fixed_size_binary(t):
        raw = np.frombuffer(arr.buffers()[1], dtype=np.uint8)
        out[name + ".bytes"] = raw[arr.offset * t.byte_width:(arr.offset + n) * t.byte_width].astype(np.float32)
    elif pa.types.is_binary(t) or pa.types.is_string(t) or pa.types.is_large_binary(t) or pa.types.is_large_string(t):
        out[name + ".len"] = pc.binary_length(arr).fill_null(0).to_numpy().astype(np.float32)
        odt = np.int64 if pa.types.is_large_binary(t) or pa.types.is_large_string(t) else np.int32
        bufs = arr.buffers()
        off = np.frombuffer(bufs[1], dtype=odt)[arr.offset:arr.offset + n + 1]
        data = np.frombuffer(bufs[2], dtype=np.uint8) if bufs[2] is not None else np.zeros(0, dtype=np.uint8)
        out[name + ".bytes"] = data[off[0]:off[-1]].astype(np.float32)
    else:                                 # fixed width: integers, floats, temporal types, decimals
        width = t.bit_width // 8
        raw = np.frombuffer(arr.buffers()[1], dtype=np.uint8)[arr.offset * width:(arr.offset + n) * width]
        if pa.types.is_floating(t):
            v = raw.view({2: np.float16, 4: np.float32, 8: np.float64}[width])
            out[name] = v.astype(np.float32 if width <= 4 else np.float64)
        elif width in (1, 2, 4) and not pa.types.is_decimal(t):
            out[name] = raw.view({1: np.int8, 2: np.int16, 4: np.int32}[width]).astype(np.float64)
        elif width == 8:
            v = raw.view(np.int64)
            out[name] = np.stack([v >> 32, v & 0xFFFFFFFF], axis=-1).astype(np.float64)
        else:
            out[name + ".bytes"] = raw.astype(np.float32)


def dump_outputs(b, w, h, directory, seed):
    """The decoded batches of result handle `h` (freed here) -> DIR/<name>.npy: `_batch_rows` (rows per output batch),
    `_sample_rows` (the rows dumped: all of them, or a sample drawn with `seed`, sorted) and every column of those rows
    through flatten_arrow.  The sample halves until the files fit in DUMP_MAX_BYTES."""
    import pyarrow as pa
    pr = b.pr
    pr._check(b.L.rv_result_to_host(h))
    batches = pr._export_batches(h.value, w["schema"])
    table = pa.Table.from_batches(batches)
    n = table.num_rows
    rows = min(n, DUMP_MAX_ROWS)
    while True:
        idx = np.sort(np.random.default_rng(seed).choice(n, rows, replace=False)) if rows < n else np.arange(n)
        sub = table.take(pa.array(idx)).combine_chunks()
        out = {"_batch_rows": np.array([x.num_rows for x in batches], dtype=np.float64), "_sample_rows": idx.astype(np.float64)}
        for name, col in zip(sub.column_names, sub.columns):
            flatten_arrow(name, col.chunk(0) if col.num_chunks == 1 else pa.concat_arrays(col.chunks), out)
        total = sum(a.nbytes for a in out.values())
        if total <= DUMP_MAX_BYTES or rows == 1:
            break
        rows //= 2
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    return {"dir": directory, "rows": int(len(idx)), "of_rows": n, "arrays": len(out), "bytes": int(total)}


def c1_line(b):
    """C1: 10 k records of the generate_avro.py schema, 8 chunks, through the Python surface the reference's README
    times (`deserialize_array_threaded(list, schema, 8)`: 1.17 ms on its author's laptop, README.md:24,30-31)."""
    import pyruhvro
    import workloads
    n, k = 10_000, 8
    sj, data, off = workloads.generate("kafka", n, seed=7)
    recs = [data[off[i]:off[i + 1]].tobytes() for i in range(n)]
    for _ in range(20):
        pyruhvro.deserialize_array_threaded(recs, sj, k)
    times = []
    for _ in range(200):
        t0 = time.perf_counter()
        out = pyruhvro.deserialize_array_threaded(recs, sj, k)
        times.append(time.perf_counter() - t0)
    assert len(out) == k and sum(x.num_rows for x in out) == n
    w = b.load("kafka", n, 7)
    dev = b.time_device(w, k, 200, 20)
    host = b.time_host(w, k, 200, 20)
    return {"workload": "C1: 10 k records, generate_avro.py schema, num_chunks = 8", "python_ms_per_call": 1000.0 * statistics.median(times),
            "python_ms_per_call_min": 1000.0 * min(times), "python_path": "pyruhvro.deserialize_array_threaded(list[bytes], schema, 8) -> 8 pyarrow.RecordBatch",
            "reference_readme_ms": 1.17, "c_abi_host_ms_per_call": host["ms_per_step"], "device_resident_ms_per_call": dev["ms_per_step"],
            "fused_kernel_ms": float(dev["kernel_ms"][0]), "records_per_s_python": n / statistics.median(times)}


def python_surface_line(b, n=1_000_000, k=8):
    """(f)2: throughput through the Python surface at a size where it matters — the list walk + pinned gather of
    `deserialize_array_threaded(list[bytes], ...)` (csrc/pymod.cpp) and the zero-copy `deserialize_arrow_array`
    (a pyarrow BinaryArray of datums), next to the C-ABI call both of them end in."""
    import pyarrow as pa
    import pyruhvro
    import workloads
    pr = b.pr
    sj, data, off = workloads.generate("kafka", n, seed=9)
    recs = [data[off[i]:off[i + 1]].tobytes() for i in range(n)]
    arr = pa.array(recs, type=pa.large_binary())

    def med(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            out = fn()
            ts.append(time.perf_counter() - t0)
        assert sum(x.num_rows for x in out) == n
        return statistics.median(ts)

    t_list = med(lambda: pyruhvro.deserialize_array_threaded(recs, sj, k))
    t_arrow = med(lambda: pr.deserialize_arrow_array(arr, sj, k))
    t_abi = med(lambda: pr.decode_packed(data, off, n, sj, k))
    return {"workload": "generate_avro.py schema, %d records, num_chunks = %d" % (n, k), "unit": UNIT,
            "list_of_bytes": n / t_list, "list_of_bytes_ms": 1000.0 * t_list,
            "arrow_binary_array": n / t_arrow, "arrow_binary_array_ms": 1000.0 * t_arrow,
            "packed_numpy_c_abi": n / t_abi, "packed_numpy_c_abi_ms": 1000.0 * t_abi,
            "note": "list_of_bytes = pyruhvro.deserialize_array_threaded (the reference's call); arrow_binary_array = deserialize_arrow_array "
                    "(no list walk, no gather); packed = decode_packed -> rv_decode_host on pageable numpy buffers"}


def config_line(b, workload, n, k, peak, peak_src, steps=10):
    w = b.load(workload, n, 42 if workload != "wide" else 43)
    dev = b.time_device(w, k, steps, 3)
    host = b.time_host(w, k, 5, 2)
    parity = parity_check(b, w, k)
    rl = b.roofline(w, dev, peak, peak_src)
    out = {"workload": WORKLOAD_DESC[workload], "records": n, "num_chunks": k, "value": n / (dev["ms_per_step"] * 1e-3), "unit": UNIT,
           "ms_per_step": dev["ms_per_step"], "input_bytes": w["total_in"], "arrow_bytes": dev["arrow_bytes"],
           "roofline_frac": rl["frac"], "path_frac": rl["path_frac"], "kernel_ms": rl["kernel_ms"],
           "e2e_value": n / (host["ms_per_step"] * 1e-3), "e2e_ms_per_step": host["ms_per_step"], "parity_checked": parity}
    del w
    b.free_pinned()
    b.torch.cuda.empty_cache()
    return out


def encode_line(b, w, k, peak):
    """The reverse direction (SURVEY.md 8(f) rank 1): Arrow -> Avro through serialize_record_batch, with its own CPU arm
    (the oracle's restatement of fast_encode.rs is pure Python, far too slow to time at this size: the ratio is against
    the decode CPU arm's bytes/s instead and says so)."""
    pr = b.pr
    n = w["n"]
    batch = pr.decode_packed(w["h_data"], w["h_off"], n, w["schema_json"], 1)[0]
    out = None
    for _ in range(3):
        out = pr.serialize_record_batch(batch, w["schema_json"], k)
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        out = pr.serialize_record_batch(batch, w["schema_json"], k)
        times.append(time.perf_counter() - t0)
    dt = statistics.median(times)
    avro_bytes = int(sum(a.nbytes for a in out))
    arrow_in = int(batch.nbytes)
    tb = (ctypes.c_float * 8)()
    km = None
    if hasattr(b.L, "rv_last_encode_timings"):
        b.L.rv_last_encode_timings.argtypes = [ctypes.POINTER(ctypes.c_float), ctypes.c_int]
        nt = b.L.rv_last_encode_timings(tb, 8)
        km = [float(tb[i]) for i in range(nt)]
    res = {"value": n / dt, "unit": UNIT, "ms_per_step": 1000.0 * dt, "path": "pyruhvro.serialize_record_batch (host Arrow in, host Avro out)",
           "avro_bytes": avro_bytes, "arrow_bytes_in": arrow_in}
    if km:
        kernel_ms = km[0] + km[1] + km[2]
        algo = arrow_in + avro_bytes + 4 * (n + k)   # reads every Arrow buffer once, writes the datum bytes + i32 offsets
        res["roofline"] = {"bound": "hbm", "kernels": "encode_size + encode_scan + encode_write", "kernel_ms": kernel_ms,
                           "size_ms": km[0], "scan_ms": km[1], "write_ms": km[2], "algorithmic_bytes": algo,
                           "achieved": algo / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0, "peak": peak, "unit": "GB/s",
                           "frac": (algo / (kernel_ms * 1e-3) / 1e9 / peak) if kernel_ms > 0 else 0.0, "h2d_ms": km[3], "d2h_ms": km[4]}
    del out, batch
    return res


def gather_mode(b, args, steps, warmup):
    """C5: every rank decodes its shard on its GPU (device-resident), then the shards' Arrow buffers are gathered into
    single RecordBatches on rank 0 over NVLink (pyruhvro_b200.distributed)."""
    import torch.distributed as dist
    from pyruhvro_b200 import distributed as D
    n_total = args.records * b.world
    r0, r1 = D.shard_bounds(n_total, b.world, b.rank)
    w = b.load(args.workload, r1 - r0, args.seed, r0=r0)
    res = None
    t_dec, t_gat = [], []
    for i in range(warmup + steps):
        res = D.decode_and_gather(w["schema_json"], w["d_data"], w["d_off"], w["n"], timing=True)
        if i >= warmup:
            t_dec.append(res["decode_ms"])
            t_gat.append(res["gather_ms"])
    dec = b.max_over_ranks(statistics.median(t_dec))
    gat = b.max_over_ranks(statistics.median(t_gat))
    if b.rank == 0:
        peak_nv = 770.0
        line = {"metric": METRIC, "value": n_total / ((dec + gat) * 1e-3), "unit": UNIT, "n_gpus": b.world, "steps": steps, "warmup": warmup,
                "ms_per_step": dec + gat, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": dict(config_of(args, b.world), mode="C5 gather: shards -> single RecordBatches on rank 0"),
                "gather": {"decode_ms": dec, "gather_ms": gat, "records_total": n_total, "batches": res["n_batches"],
                           "gathered_bytes": res["gathered_bytes"], "nvlink_bytes_into_rank0": res["remote_bytes"],
                           "nvlink_gbs": res["remote_bytes"] / max(gat * 1e-3, 1e-9) / 1e9, "nvlink_peak_gbs": peak_nv,
                           "nvlink_frac": res["remote_bytes"] / max(gat * 1e-3, 1e-9) / 1e9 / peak_nv,
                           "how": res["how"]},
                "gpu_launches": res["launches"]}
        print(json.dumps(line), flush=True)
    if b.world > 1:
        dist.barrier(device_ids=[b.local_rank])


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # convenience: re-launch under torchrun the way the driver does
        import subprocess
        port = os.environ.get("MASTER_PORT", "29517")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", port, os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    steps, warmup = args.steps, max(3, args.warmup)

    if args.impl == "reference":
        if rank == 0:
            cpu_arm(args, steps, warmup, emit_line=True, world=world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the decode path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = bind_to_gpu_node(torch, local_rank) if world > 1 else None   # one rank per GPU: each on its GPU's socket
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    b = Bench(args, rank, local_rank, world)

    if args.gather:
        gather_mode(b, args, steps, warmup)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- workload: this rank's shard, generated straight into pinned host memory ----------
    n, k = args.records, args.num_chunks
    w = b.load(args.workload, n, args.seed, r0=rank * n)
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    # the line carries rank 0's clocks; the other ranks do not poll NVML (eight pollers contend on the driver for nothing)
    sampler = ClockSampler(int(vis.split(",")[local_rank]) if vis else local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    dump = args.dump_outputs if rank == 0 else None   # rank 0's shard: the first `records` rows
    dev_res = b.time_device(w, k, steps, warmup, sampler, keep_last=bool(dump))
    dumped = dump_outputs(b, w, dev_res.pop("last"), dump, args.seed) if dump else None
    host_res = b.time_host(w, k, steps, warmup, sampler)
    if sampler:
        sampler.stop()
    value = world * n / (dev_res["ms_per_step"] * 1e-3)
    e2e_value = world * n / (host_res["ms_per_step"] * 1e-3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = hbm_peak()
    rl = b.roofline(w, dev_res, peak, peak_src)
    rl["traffic"], rl["traffic_capture"] = traffic_of(args.workload, n)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": dev_res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "config": config_of(args, world),
        "bytes": {"input_per_gpu": w["total_in"], "offsets_per_gpu": 8 * (n + 1), "arrow_per_gpu": dev_res["arrow_bytes"]},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": host_res["h2d_bytes"], "d2h_bytes_per_step": host_res["d2h_bytes"],
                "ms_per_step": host_res["ms_per_step"], "h2d_busy_ms": host_res["h2d_busy_ms"], "d2h_busy_ms": host_res["d2h_busy_ms"],
                "h2d_gbs_while_copying": host_res["h2d_gbs_while_copying"], "d2h_gbs_while_copying": host_res["d2h_gbs_while_copying"],
                "per_rank": host_res["per_rank"],
                "path": "rv_decode_host: pinned host Avro in -> pinned host Arrow out, chunks pipelined on persistent NUMA-bound workers"},
        "gpu_launches": dev_res["launches"],
        "roofline": rl,
        "clocks": sampler.summary() if sampler else None,
    }
    if dumped:
        line["dumped_outputs"] = dumped
    if world > 1:
        line["rank_binding"] = {"rank0_numa_node": numa_node, "how": "each rank's threads run on the CPUs of its GPU's NUMA node (bench.py: bind_to_gpu_node)"}
    if world == 1 and not args.no_extras:
        try:
            line["parity_checked"] = parity_check(b, w, k)
        except AssertionError as e:
            line["parity_checked"] = False
            line["parity_error"] = str(e)[:300]
        try:
            line["encode"] = encode_line(b, w, k, peak)
        except Exception as e:  # pragma: no cover
            line["encode"] = {"error": str(e)[:200]}
        del w
        b.free_pinned()
        torch.cuda.empty_cache()
        for key, fn in (("c1", lambda: c1_line(b)), ("python_surface", lambda: python_surface_line(b)), ("c2", lambda: config_line(b, "flat", n, k, peak, peak_src)),
                        ("c4", lambda: config_line(b, "wide", n, k, peak, peak_src))):
            try:
                line[key] = fn()
            except Exception as e:  # pragma: no cover
                line[key] = {"error": (type(e).__name__ + ": " + str(e))[:300]}
            b.free_pinned()
        line["cpu_baseline"] = cpu_arm(args, steps=5, warmup=1, emit_line=False)
    print(json.dumps(line), flush=True)
    b.free_pinned()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
