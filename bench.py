#!/usr/bin/env python3
"""bench.py -- Nexmark-shaped streaming HashJoin (headline) and HashAgg (secondary) throughput.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--legs value,e2e,agg,chain,cpu] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], "Nexmark q7/q8 streaming HashJoin (bid x auction) 1xB200, 10M build
rows in HBM"; SURVEY 8(d) cfg3):  the auction side (10 000 000 rows: id, seller, category, expires)
is loaded into the right-side join state, then every STEP pushes one batch of 2^20 bid rows
(auction, date_time, bidder, price; 1024 StreamChunks of 1024 rows coalesced into one device batch)
through the inner-join operator: each bid probes the auction state (1 match), the joined 8-column
rows are emitted, and the bid is inserted into the left-side state.  metric = input rows / s.
N > 1 (configs[3]): every rank generates its own bid / auction shard; a step partitions the bids by the
reference's CRC32 vnode on the GPU, stores them straight into the owning rank's receive region over
NVLink peer memory (one library call, device barrier), and the join consumes the received rows with
the row count read on the device -- weak scaling: 10M build rows and 2^20 bid rows per step PER GPU.
RWGPU_EXCHANGE=nccl selects partition + NCCL all-to-all-v instead.

`value`   : inputs already resident in HBM, `rwgpu_join_push_device` (CUDA-event timed, max over ranks).
`e2e`     : the same steps through the host-buffer C-ABI call `rwgpu_join_push` (pinned host chunks in,
            host output chunk views out; H2D / D2H inside the timed region; N>1: host input partitioned
            per rank, no exchange).
`secondary`: BASELINE configs[1] (q4-shaped HashAgg: count(*), sum, max GROUP BY auction, 2^18-row epochs).
`chain`   : join -> Filter -> Project -> HashAgg without leaving HBM (SURVEY 8(f) rank 1), a barrier per batch.
`roofline`: dominant kernel, algorithmic bytes / CUDA-event time against MEASURED_PEAKS.json; `traffic` from the
            committed ncu capture (profiles/r1_traffic.json).  `clocks`: in-process NVML samples during the region.
`--impl reference`: the CPU restatement of the reference algorithm (oracle/fastcpu.cc, one
single-threaded actor per host core, inputs pre-partitioned by vnode) on a bounded sample.
`--dump-outputs DIR`: after the timed steps, the join output of the last one as DIR/<name>.npy (see dump_outputs), so
that two builds can be compared output for output: the inputs are generated from fixed seeds.
"""
import argparse
import contextlib
import io
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (which may be read-only)

N_BUILD = 10_000_000
BATCH = 1 << 20
CHUNK = 1024
SEED = 0x20210410
AGG_EPOCH_ROWS = 1 << 18
AGG_KEYS = 1 << 20
AGG_SEED = 0x20210401

# algorithmic bytes per input row (SURVEY 8(d)); see DESIGN.md "Roofline arithmetic"
JOIN_BYTES_PER_ROW_STEP = 194.125    # probe + emit + own-side insert, m = 1
JOIN_BYTES_PER_ROW_PROBE = 146.125   # dominant kernel only: W_u + 1.125 + S + m*(W_m + W_out + 1)
AGG_BYTES_PER_ROW_FLOOR = 73.125     # W_in + 1.125 + K + 2A


# ------------------------------------------------------------------------------------------ data
def splitmix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    z = x
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def gen_auctions(n, seed, id_base=0):
    """auction rows in a pseudo-random arrival order: (id, seller, category, expires)."""
    with np.errstate(over="ignore"):
        i = np.arange(n, dtype=np.uint64)
        order = np.argsort(splitmix64(i ^ np.uint64(seed)), kind="stable")
        ids = (order.astype(np.int64) + id_base)
        seller = (splitmix64(i ^ np.uint64(seed + 1)) % np.uint64(1_000_000)).astype(np.int64)
        category = (np.uint64(10) + splitmix64(i ^ np.uint64(seed + 2)) % np.uint64(5)).astype(np.int64)
        expires = (splitmix64(i ^ np.uint64(seed + 3)) % np.uint64(1 << 40)).astype(np.int64)
    return [ids, seller, category, expires]


def gen_bids(n, start, seed, n_auction, id_base=0, hot=False):
    """bid rows (auction, date_time [unique, the stream key], bidder, price).  hot: with p = 1/2 a bid goes to one of the
    last 100 auction ids (SURVEY 8(d) cfg3 "hot" variant, the Nexmark hot-auction shape)."""
    with np.errstate(over="ignore"):
        i = np.arange(start, start + n, dtype=np.uint64)
        auction = (splitmix64(i ^ np.uint64(seed + 10)) % np.uint64(n_auction)).astype(np.int64) + id_base
        if hot:
            h = splitmix64(i ^ np.uint64(seed + 13))
            is_hot = (h & np.uint64(1)) == np.uint64(1)
            hot_id = (n_auction - 100 + ((h >> np.uint64(8)) % np.uint64(100)).astype(np.int64)) + id_base
            auction = np.where(is_hot, hot_id, auction)
        date_time = i.astype(np.int64) + 1_600_000_000_000_000
        bidder = (splitmix64(i ^ np.uint64(seed + 11)) % np.uint64(1_000_000)).astype(np.int64)
        price = (splitmix64(i ^ np.uint64(seed + 12)) % np.uint64(1 << 24)).astype(np.int64)
    return [auction, date_time, bidder, price]


def gen_agg_rows(n, start, seed, hot=False):
    """(auction key, price).  hot = SURVEY 8(d) cfg2 dist B: with p = 1/2 the key is one of 128 hot auctions."""
    with np.errstate(over="ignore"):
        i = np.arange(start, start + n, dtype=np.uint64)
        key = (splitmix64(i ^ np.uint64(seed)) % np.uint64(AGG_KEYS)).astype(np.int64)
        if hot:
            h = splitmix64(i ^ np.uint64(seed + 3))
            key = np.where((h & np.uint64(1)) == np.uint64(1), ((h >> np.uint64(8)) % np.uint64(128)).astype(np.int64), key)
        price = (splitmix64(i ^ np.uint64(seed + 7)) % np.uint64(1 << 24)).astype(np.int64)
    return [key, price]


def gen_auction_updates(auct, lo, n_pairs):
    """U-/U+ pairs for auctions lo .. lo+n_pairs-1 of the arrival order: the stored row retracted, the same id
    re-inserted with a new `expires` (SURVEY 8(d) cfg3 retraction phase).  -> (ops, cols) of 2 * n_pairs rows."""
    ops = np.tile(np.array([4, 3], np.uint8), n_pairs)
    cols = []
    for k, c in enumerate(auct):
        old = c[lo:lo + n_pairs]
        new = old + 1 if k == 3 else old
        cols.append(np.ascontiguousarray(np.stack([old, new], 1).reshape(-1)))
    return ops, cols


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  In-process NVML (what nvidia-smi
    itself reads) every 2 ms: spawning `nvidia-smi -lms` next to a timed region that lasts a few
    milliseconds put its start-up (driver attach) inside the measurement and stalled kernel launches
    for milliseconds.  nvidia-smi is the fallback when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index=0):
        self.idx = gpu_index
        self.proc = None
        self.nv = None
        self.samples = []
        self.thread = None
        self.halt = False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.halt:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((float(sm), int(rs)))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            import threading
            self.halt = False
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        self.path = tempfile.mktemp(suffix=".csv")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.nv is not None:
            self.halt = True
            if self.thread is not None:
                self.thread.join(timeout=2)
            if not self.samples:  # region shorter than one sampling period: take one sample now
                try:
                    self.samples.append((float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)), 0))
                except Exception:
                    pass
            sm = [x[0] for x in self.samples]
            bits = 0
            for x in self.samples:
                bits |= x[1]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(name for bit, name in self.REASONS if bits & bit), "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def pin_to_gpu_numa_node(gpu_index):
    """Run this process (and first-touch its pinned buffers) on the CPU socket the GPU hangs off: host<->device
    copies that cross the socket interconnect lose a third of their bandwidth.  Deployment detail of any
    GPU-attached worker, not part of the measured path; a failure here is ignored."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu captures (profiles/r2_traffic.json, r1_traffic.json), or None"""
    for f in ("r2_traffic.json", "r1_traffic.json"):
        try:
            return float(json.load(open(os.path.join(ROOT, "profiles", f)))[kernel]["bytes_per_launch"])
        except Exception:
            continue
    return None


def bench_config(world):
    """the `config` object of the JSON line -- key-identical in both arms (the driver compares them)"""
    return {"workload": "nexmark_q7q8_hashjoin_cfg3" if world == 1 else "nexmark_q8_shuffled_hashjoin_cfg4",
            "build_rows_per_gpu": N_BUILD, "probe_rows_per_step_per_gpu": BATCH, "chunk_rows": CHUNK}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ CPU arm
class FastCpu:
    def __init__(self):
        p = os.path.join(ROOT, "oracle", "_build", "libfastcpu.so")
        if not os.path.exists(p):
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
        f = C.CDLL(p)
        f.rwf_join_new.restype = C.c_void_p
        f.rwf_join_free.argtypes = [C.c_void_p]
        f.rwf_join_reserve.argtypes = [C.c_void_p, C.c_int, C.c_uint64]
        f.rwf_join_push.restype = C.c_int64
        f.rwf_join_push.argtypes = [C.c_void_p, C.c_int, C.c_int64] + [C.c_void_p] * 5
        f.rwf_agg_new.restype = C.c_void_p
        f.rwf_agg_new.argtypes = [C.c_int]
        f.rwf_agg_free.argtypes = [C.c_void_p]
        f.rwf_agg_reserve.argtypes = [C.c_void_p, C.c_uint64]
        f.rwf_agg_push.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        f.rwf_agg_flush.restype = C.c_int64
        f.rwf_agg_flush.argtypes = [C.c_void_p]
        self.f = f


def vnode_of_int64(keys):
    """crc32(8 LE bytes) % 256 per key (vnode.rs:45-50) -- numpy table-driven, used to pre-partition
    the CPU arm's input the way HashDataDispatcher would deliver it."""
    tab = np.zeros(256, dtype=np.uint32)
    for i in range(256):
        c = i
        for _ in range(8):
            c = (0xEDB88320 ^ (c >> 1)) if (c & 1) else (c >> 1)
        tab[i] = c
    crc = np.full(len(keys), 0xFFFFFFFF, dtype=np.uint32)
    u = keys.astype(np.uint64)
    for b in range(8):
        byte = ((u >> np.uint64(8 * b)) & np.uint64(0xFF)).astype(np.uint32)
        crc = tab[(crc ^ byte) & 0xFF] ^ (crc >> 8)
    return ((crc ^ 0xFFFFFFFF) % 256).astype(np.int32)


CHECKSUM_WEIGHTS = (3, 31, 5, 7, 11, 1, 17, 19)  # oracle/fastcpu.cc OutBuilder::append

DUMP_COLUMNS = ("bid_auction", "bid_date_time", "bid_bidder", "bid_price", "auction_id", "auction_seller", "auction_category",
                "auction_expires")
DUMP_MAX_ROWS = 1 << 19  # 8 float64 columns + float32 ops: ~36 MB
DUMP_SEED = 0x5EED


def dump_outputs(out_dir, view):
    """Writes the output view of a join push as out_dir/<name>.npy.  The visible rows are sorted by all columns (the row
    order of a join's output is not part of its result) and a fixed, seeded sample of at most DUMP_MAX_ROWS of them is kept:
    ops.npy (float32) and one float64 array per output column (exact: every value of the workload is below 2^53).
    summary.npy covers ALL visible rows: [row count, low and high 32 bits of the order-independent checksum of
    DeviceView.checksum(CHECKSUM_WEIGHTS)]."""
    os.makedirs(out_dir, exist_ok=True)
    ops = view.ops().cpu().numpy()
    cols = [view.column(k).cpu().numpy() for k in range(view.n_cols)]
    vis = view.visible()
    if vis is not None:
        keep = vis.cpu().numpy()
        ops, cols = ops[keep], [c[keep] for c in cols]
    order = np.lexsort([ops] + cols[::-1])  # primary key: column 0
    n = len(ops)
    if n > DUMP_MAX_ROWS:
        order = order[np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MAX_ROWS, replace=False))]
    rows, cs = view.checksum(CHECKSUM_WEIGHTS)
    np.save(os.path.join(out_dir, "summary.npy"), np.array([rows, cs & 0xFFFFFFFF, cs >> 32], np.float64))
    np.save(os.path.join(out_dir, "ops.npy"), ops[order].astype(np.float32))
    for name, c in zip(DUMP_COLUMNS, cols):
        np.save(os.path.join(out_dir, name + ".npy"), c[order].astype(np.float64))


def cpu_topology():
    """-> (allowed logical CPUs, one logical CPU per physical core among them, cgroup CPU quota or None)."""
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    seen, phys = set(), []
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            phys.append(c)
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            f = open(path).read().split()
            if path.endswith("cpu.max"):
                if f[0] != "max":
                    quota = float(f[0]) / float(f[1])
            else:
                q = float(f[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except (OSError, ValueError, IndexError):
            continue
    return allowed, phys, quota


class CpuActors:
    """P = len(cpu_ids) single-threaded actors (oracle/fastcpu.cc rwf_pool_*: one long-lived OS thread each, pinned to
    cpu_ids[a], tables first-touched on that thread), input vnode-partitioned the way HashDataDispatcher would deliver
    it, each actor consuming ITS stream of 1024-row chunks independently."""

    def __init__(self, cpu_ids, pin=True, chunk=CHUNK):
        fc = FastCpu().f
        self.fc, self.P, self.chunk, self.pin = fc, len(cpu_ids), chunk, pin
        fc.rwf_pool_new.restype = C.c_void_p
        fc.rwf_pool_new.argtypes = [C.c_int, C.c_void_p]
        fc.rwf_pool_reserve.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        fc.rwf_pool_run.restype = C.c_int64
        fc.rwf_pool_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p]
        fc.rwf_pool_pin_failures.argtypes = [C.c_void_p]
        fc.rwf_pool_checksum.restype = C.c_uint64
        fc.rwf_pool_checksum.argtypes = [C.c_void_p]
        fc.rwf_pool_free.argtypes = [C.c_void_p]
        ids = np.asarray(cpu_ids if pin else [-1] * self.P, dtype=np.int32)
        self.pool = fc.rwf_pool_new(self.P, ids.ctypes.data)

    def pack(self, blist):
        """vnode-partition every batch (a batch is `cols` = all-Insert, or `(ops, cols)`); -> argument arrays indexed
        [batch * P + actor] (+ keepalive)"""
        P, nb = self.P, len(blist)
        cnts = np.zeros((nb, P), np.int64)
        ptrs = [(C.c_void_p * (nb * P))() for _ in range(5)]
        keep = []
        for b, item in enumerate(blist):
            ops_in, cols = item if isinstance(item, tuple) else (None, item)
            part = vnode_of_int64(cols[0]) * P // 256
            order = np.argsort(part, kind="stable")
            cnt = np.bincount(part, minlength=P).astype(np.int64)
            off = np.concatenate([[0], np.cumsum(cnt)[:-1]])
            sc = [np.ascontiguousarray(c[order]) for c in cols]
            ops = np.ones(len(order), np.uint8) if ops_in is None else np.ascontiguousarray(ops_in[order])
            keep.append((ops, sc))
            cnts[b] = cnt
            for a in range(P):
                ptrs[0][b * P + a] = ops.ctypes.data + int(off[a])
                for k in range(4):
                    ptrs[1 + k][b * P + a] = sc[k].ctypes.data + int(off[a]) * 8
        return nb, cnts, ptrs, keep

    def reserve(self, build_cols):
        """size every actor's tables for its share of the build side's keys, on the actor's own thread"""
        part = vnode_of_int64(build_cols[0]) * self.P // 256
        keys = np.ascontiguousarray(np.bincount(part, minlength=self.P).astype(np.uint64))
        self.fc.rwf_pool_reserve(self.pool, keys.ctypes.data, keys.ctypes.data)

    def run(self, side, batches, warmup=0):
        """-> dict(value = rows/s over the batches after the first `warmup`, out_rows / checksum of those, ...)"""
        fc, P = self.fc, self.P
        nb, cnts, ptrs, keep = self.pack(batches)
        cs0 = None
        if warmup:  # the checksum is cumulative: run the warm-up batches in a call of their own
            self._call(side, (warmup, cnts[:warmup], [self._slice(p, 0, warmup) for p in ptrs]), 0)
        cs0 = fc.rwf_pool_checksum(self.pool)
        out_rows, wall, busy = self._call(side, (nb - warmup, cnts[warmup:], [self._slice(p, warmup, nb) for p in ptrs]), 0)
        rows = sum(len((b[1] if isinstance(b, tuple) else b)[0]) for b in batches[warmup:])
        return {"value": rows / wall if wall > 0 else 0.0, "wall_s": wall, "actors": P, "busy_s_min": float(busy.min()),
                "busy_s_max": float(busy.max()), "busy_s_mean": float(busy.mean()),
                "pin_failures": int(fc.rwf_pool_pin_failures(self.pool)) if self.pin else None, "out_rows": out_rows,
                "checksum": (fc.rwf_pool_checksum(self.pool) - cs0) & ((1 << 64) - 1)}

    def _slice(self, arr, lo, hi):
        n = (hi - lo) * self.P
        out = (C.c_void_p * max(n, 1))()
        for i in range(n):
            out[i] = arr[lo * self.P + i]
        return out

    def _call(self, side, packed, warm):
        nb, cnts, ptrs = packed
        cnts = np.ascontiguousarray(cnts)
        wall = C.c_double()
        busy = np.zeros(self.P, np.float64)
        rows = self.fc.rwf_pool_run(self.pool, side, nb, warm, cnts.ctypes.data, *ptrs, self.chunk, C.byref(wall), busy.ctypes.data)
        return int(rows), wall.value, busy

    def close(self):
        if self.pool:
            self.fc.rwf_pool_free(self.pool)
            self.pool = None


def cpu_join_run(auct, batches, cpu_ids, warmup, chunk=CHUNK, pin=True, after=None):
    """build side `auct` (untimed), then the probe-side `batches` (the first `warmup` untimed) through P pinned actors;
    `after` = optional (side, batches) pushed afterwards, its result under key "after".  -> dict (see CpuActors.run)"""
    ca = CpuActors(cpu_ids, pin, chunk)
    ca.reserve(auct)
    ca.run(1, [auct])
    res = ca.run(0, batches, warmup)
    if after is not None:
        res["after"] = ca.run(after[0], after[1])
    ca.close()
    return res


# ------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from risingwave_b200 import abi, device
    from risingwave_b200.executor import AggCall, Backend, HashAggExecutor, HashJoinExecutor, JoinParams, MockSource
    from risingwave_b200.stream_chunk import Column, StreamChunk

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    pin_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # create the NCCL communicator NOW: the first collective builds it lazily (~0.3 s), and with the
        # peer-memory exchange the first collective would otherwise be the barrier that opens the timed region
        warm = torch.zeros(1, device="cuda")
        dist.all_reduce(warm)
        dist.barrier()
        torch.cuda.synchronize()
    be = Backend.cuda()
    K, W = args.steps, args.warmup
    legs = set(args.legs.split(","))
    T4 = [abi.T_INT64] * 4
    stream = torch.cuda.Stream()
    peak, which = measured_peak_hbm()

    def new_join():
        _, sl = MockSource.channel()
        _, sr = MockSource.channel()
        # left = bid (key col 0, stream key date_time), right = auction (key col 0 = id = stream key)
        return HashJoinExecutor(be, abi.JOIN_INNER, sl.into_executor(T4, [1]), sr.into_executor(T4, [0]),
                                JoinParams([0], [1]), JoinParams([0], []), [False],
                                capacity_hint=(N_BUILD, N_BUILD),  # distinct auction ids per GPU, both sides
                                stored_rows_hint=(int((K + W + V + 4) * BATCH * 1.12) + 6 * world * BATCH, 0))  # bids this GPU will store (its share:
        # ~BATCH per step) + the upper bounds of the pushes in flight (a counted push reserves for its buffer's capacity)
        # (the bid side is sized for the run: at 6 G rows/s it grows by ~290 GB/s, three times faster than cudaMalloc hands
        #  out memory -- 200 MB in 1.5-2 ms; a helper thread keeps one 200 MB segment ahead for streams that grow at a
        #  realistic rate, DESIGN 4.2)

    def to_dev(cols):
        return [torch.from_numpy(c).cuda() for c in cols]

    def dchunk(cols_dev):
        n = cols_dev[0].numel()
        return device.DeviceChunk(torch.ones(n, dtype=torch.uint8, device="cuda"), cols_dev, T4)

    id_base = rank * N_BUILD
    auct = gen_auctions(N_BUILD, SEED + rank * 1000, id_base)
    # bids of rank r reference auctions of ALL ranks (so the shuffle really moves rows)
    V = 2  # verification batches pushed AFTER the timed region and compared with the CPU restatement (checksum + row count)
    bid_start = lambda r, s: (r * (K + W + V) + s) * BATCH  # noqa: E731  (disjoint date_time ranges per rank)
    batches_host = [gen_bids(BATCH, bid_start(rank, s), SEED, N_BUILD * world) for s in range(K + W + V)]

    if world > 1:
        from risingwave_b200 import exchange
        ex_kind = os.environ.get("RWGPU_EXCHANGE", "flat")
        if ex_kind == "nccl":
            ex_plan = exchange.ShufflePlan(world, rank, key_indices=[0], types=T4)
            ex_name = "crc32 vnode partition kernel + NCCL all_to_all_single per column"
        elif ex_kind == "p2p":
            ex_plan = exchange.P2PShufflePlan(world, rank, key_indices=[0], types=T4, batch_rows=BATCH)
            ex_name = "crc32 vnode partition kernel storing straight into the peers' receive regions over NVLink (symmetric memory), device barrier, unpack kernel"
        else:
            ex_plan = exchange.FlatShufflePlan(world, rank, key_indices=[0], types=T4, batch_rows=BATCH,
                                               max_blocks=int(os.environ.get("RWGPU_EXCHANGE_BLOCKS", "0")))
            ex_name = ("one kernel per batch: crc32 vnode histograms, scan, count exchange + cross-rank barrier, scatter over NVLink "
                       "(symmetric memory) into the rows' final place in the destination's receive buffer, barrier; the join reads the buffer in place")

    def shuffled(cols_dev):
        if world == 1:
            return dchunk(cols_dev)
        ops, cols = ex_plan.exchange(dchunk(cols_dev), stream)
        return device.DeviceChunk(ops, cols, T4)

    line = {}
    verify_gpu = retract_verify = hot_verify = None
    with torch.cuda.stream(stream):
        auct_dev = to_dev(auct)

        build_first_ms = [0.0]

        def build(join, shuffle=True):
            """-> seconds per build row, measured over the pushes AFTER the first one (the first push allocates the handle's
            output set and scratch -- tens of milliseconds of cudaMalloc, reported separately)"""
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            t1, rows_timed = t0, 0
            for i in range(0, N_BUILD, BATCH):
                part = [c[i:i + BATCH] for c in auct_dev]
                device.join_push_device(join, abi.SIDE_RIGHT, shuffled(part) if shuffle else dchunk(part), stream)
                if i == 0:
                    torch.cuda.synchronize()
                    t1 = time.perf_counter()
                    build_first_ms[0] = 1e3 * (t1 - t0)
                else:
                    rows_timed += part[0].numel()
            torch.cuda.synchronize()
            return (time.perf_counter() - t1) / max(rows_timed, 1)

        # ================================================================ leg: value (device-resident)
        if "value" in legs:
            join = new_join()
            build_s = build(join)
            batches_dev = [to_dev(b) for b in batches_host[:K + W]]
            torch.cuda.synchronize()

            # N=1: the step's input is the resident batch; N>1: the exchange is part of the step
            chunks_dev = [dchunk(b) for b in batches_dev]
            torch.cuda.synchronize()

            trace = os.environ.get("BENCH_TRACE") is not None  # per-phase wall clock (adds syncs: never for a reported number)

            counted = world > 1 and isinstance(ex_plan, (exchange.P2PShufflePlan, exchange.FlatShufflePlan))
            # the join sizes its bookkeeping (row-id and key upper bounds, output area) for the CAPACITY of a counted push; a
            # rank receives ~BATCH rows per step, so the view handed to the join covers min(world, 4) x BATCH rows of the
            # world x BATCH receive buffer (a step with more rows than that fails loudly: JERR_BAD_COUNT)
            def recv_view(b):
                ops_b, cols_b = ex_plan.output(b)
                m = min(ops_b.numel(), min(world, 4) * BATCH)
                return device.DeviceChunk(ops_b[:m], [c[:m] for c in cols_b], T4)

            recv_chunks = [recv_view(b) for b in range(2)] if counted else None
            t_ex = t_join = 0.0
            pending = {}
            lookahead = True
            # (BENCH_EX_PRIO=1: the exchange on a high-priority stream -- its blocks get the SM slots the join's kernel frees)
            ex_stream = (torch.cuda.Stream(priority=-1) if os.environ.get("BENCH_EX_PRIO") else torch.cuda.Stream()) if counted else None

            join_done = {}
            keep = {}

            def launch(s):
                """LAUNCH half of step s: (N>1) the exchange, then the push -- everything is only enqueued"""
                nonlocal t_ex, t_join
                if counted:
                    # N>1: the exchange of batch s+1 is enqueued (its own stream) before the join of batch s is launched;
                    # the join waits for its exchange ON THE DEVICE (event) and reads the received row count there
                    # (n_rows_dev).  Receive buffer b = s & 1 is reused by exchange s+2, which therefore waits (on the
                    # device) for the join of batch s.
                    ta = time.perf_counter()
                    for t in (s, s + 1):
                        if t in pending or t >= len(chunks_dev) or (t == s + 1 and (not lookahead or t == W)):
                            continue  # (nothing of the timed region starts before e0)
                        if t - 2 in join_done:
                            ex_stream.wait_event(join_done.pop(t - 2))
                        pending[t] = ex_plan.start(chunks_dev[t], ex_stream)
                    b = pending.pop(s)
                    stream.wait_event(ex_plan.events[b])
                    tb = time.perf_counter()
                    device.join_push_device_async(join, abi.SIDE_LEFT, recv_chunks[b], stream, n_rows_dev=ex_plan.count_ptr(b))
                    ev = torch.cuda.Event()
                    ev.record(stream)
                    join_done[s] = ev
                    t_ex += tb - ta
                    t_join += time.perf_counter() - tb
                    return
                ch = chunks_dev[s] if world == 1 else device.DeviceChunk(*ex_plan.exchange(chunks_dev[s], stream), T4)
                keep[s] = ch  # the input buffers stay alive until the push is collected
                device.join_push_device_async(join, abi.SIDE_LEFT, ch, stream)

            def collect(s):
                nonlocal t_join
                tb = time.perf_counter()
                out = device.join_collect(join, stream)
                t_join += time.perf_counter() - tb
                keep.pop(s, None)
                return out

            tl = []  # BENCH_TRACE: host timeline (never for a reported number)
            last_out = [None]  # output view of the last step run (valid until the next push reuses its output set)

            def run_steps(lo, hi, each=None):
                """steps lo..hi-1, push s+1 launched before push s is collected (two output sets)"""
                tot = 0
                for s in range(lo, hi):
                    t_a = time.perf_counter()
                    launch(s)
                    t_b = time.perf_counter()
                    if s > lo:
                        o = collect(s - 1)
                        tot += o.n_rows
                        if each:
                            each(o)
                    if trace:
                        tl.append((s, 1e3 * (t_b - t_a), 1e3 * (time.perf_counter() - t_b)))
                o = collect(hi - 1)
                tot += o.n_rows
                last_out[0] = o
                if each:
                    each(o)
                return tot

            sampler = ClockSampler(local_rank)
            run_steps(0, W)
            device.profile(join, "join", True)
            l0 = device.launches(join, "join")
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            if rank == 0:
                sampler.start()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            t_ex = t_join = 0.0
            out_rows = run_steps(W, W + K)
            e1.record(stream)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ms = e0.elapsed_time(e1)
            if trace:
                print("[trace] step: launch ms, collect(prev) ms\n" + "\n".join(f"  {a}: {b:.3f} {c:.3f}" for a, b, c in tl[-K:]), file=sys.stderr)
            clocks = sampler.stop() if rank == 0 else None
            kern_ms, kern_n = device.profile(join, "join", False)
            launches = device.launches(join, "join") - l0
            if args.dump_outputs and rank == 0:  # (before the verification pushes reuse the output sets)
                dump_outputs(args.dump_outputs, last_out[0])
            if world > 1:
                t = torch.tensor([ms], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
                orow = torch.tensor([out_rows], device="cuda", dtype=torch.int64)
                dist.all_reduce(orow)
                out_rows = int(orow.item())
            rows_total = K * BATCH * world
            fused_gbs = JOIN_BYTES_PER_ROW_STEP * BATCH * kern_n / (kern_ms / 1e3) / 1e9 if kern_ms else None
            line.update({
                "metric": "Nexmark q7/q8-shaped streaming HashJoin input rows/s", "value": rows_total / (ms / 1e3), "unit": "rows/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": bench_config(world),
                "config_detail": {"chunks_coalesced_per_launch": BATCH // CHUNK,
                                  "join": "inner bid.auction = auction.id, Key64, 4+4 int64 cols, 8 out cols",
                                  "l2": "inputs_larger_than_l2 (fresh 32 MiB batch per step; >1.3 GB of join state)",
                                  "exchange": None if world == 1 else ex_name},
                "host_ms_per_step": {"enqueue_exchange": 1e3 * t_ex / K, "join_launch_and_collect": 1e3 * t_join / K},
                "build_rows_per_s": world / build_s, "build_first_push_ms": build_first_ms[0], "out_rows": out_rows, "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "hbm", "kernel": "uni_hot_kernel<false,false,4> (unified bucket: probe + emit + own-side append, 4 lanes per row)",
                             "achieved": fused_gbs, "peak": peak, "unit": "GB/s", "frac": fused_gbs / peak if fused_gbs else None,
                             "traffic": ncu_traffic("uni_hot_kernel"), "traffic_unit": "bytes per launch (ncu dram read+write)",
                             "algorithmic_bytes_per_launch": JOIN_BYTES_PER_ROW_STEP * BATCH,
                             "peak_source": which, "algorithmic_bytes_per_row": JOIN_BYTES_PER_ROW_STEP,
                             "rows_per_launch": BATCH, "kernel_ms_avg": kern_ms / max(kern_n, 1),
                             "kernel_share_of_step": kern_ms / ms if ms else None}})
            # ---- verification (outside the timed region): V more batches through the SAME path (exchange included at
            # N>1) on the bench-scale state; the (row count, order-independent checksum) of their output is compared
            # below with the CPU restatement fed the same rows.
            if not os.environ.get("BENCH_NO_VERIFY"):
                vr = vc = 0
                for v in range(V):
                    chunks_dev.append(dchunk(to_dev(batches_host[K + W + v])))

                def add_checksum(o):
                    nonlocal vr, vc
                    rows_v, cs_v = o.checksum(CHECKSUM_WEIGHTS)
                    vr += rows_v
                    vc = (vc + cs_v) & ((1 << 64) - 1)

                for v in range(V):  # (one at a time: the checksum reads the view before the next push reuses the set)
                    run_steps(K + W + v, K + W + v + 1, add_checksum)
                if world > 1:
                    t = torch.tensor([vr, vc & 0xffffffff, vc >> 32], device="cuda", dtype=torch.int64)
                    dist.all_reduce(t)
                    vr, vc = int(t[0].item()), (int(t[1].item()) + (int(t[2].item()) << 32)) & ((1 << 64) - 1)
                verify_gpu = (vr, vc)
            # ================================================================ leg: retract (SURVEY 8(d) cfg3 retraction phase)
            # the same handle, now holding (W + K + V) x 2^20 bids: auction UPDATES (U- stored row / U+ same id, new
            # `expires`) probe the bid side -- every matched bid is emitted twice (- then +), the first time multi-match
            # emission, the own-side delete kernel and re-insertion are timed.  Step = 2^19 pairs = 2^20 rows.
            if "retract" in legs and world == 1:
                RP, KR, WR = 1 << 19, 8, 2  # (2 warm-up steps: each output set grows once to hold ~3 output rows per input row)
                ups = [gen_auction_updates(auct, s * RP, RP) for s in range(WR + KR + 1)]  # (+1: verification step)
                ups_dev = [device.DeviceChunk(torch.from_numpy(o).cuda(), to_dev(c), T4) for o, c in ups]
                torch.cuda.synchronize()

                def run_updates(lo, hi, each=None):
                    tot = 0
                    for s in range(lo, hi):
                        device.join_push_device_async(join, abi.SIDE_RIGHT, ups_dev[s], stream)
                        if s > lo:
                            o = device.join_collect(join, stream)
                            tot += o.n_rows
                        if each and s > lo:
                            each(o)
                    o = device.join_collect(join, stream)
                    tot += o.n_rows
                    if each:
                        each(o)
                    return tot

                run_updates(0, WR)
                device.profile(join, "join", True)
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                r0.record(stream)
                r_out = run_updates(WR, WR + KR)
                r1.record(stream)
                torch.cuda.synchronize()
                rms = r0.elapsed_time(r1)
                rk_ms, rk_n = device.profile(join, "join", False)
                cs = [0, 0]

                def add_cs(o):
                    a, b = o.checksum(CHECKSUM_WEIGHTS)
                    cs[0] += a
                    cs[1] = (cs[1] + b) & ((1 << 64) - 1)

                run_updates(WR + KR, WR + KR + 1, add_cs)
                retract_verify = (cs[0], cs[1], ups[:WR + KR], ups[WR + KR])
                m_avg = r_out / (KR * 2 * RP)  # visible + filler rows per input row (upper bound of matches per row)
                bpr = 33.125 + 16 + m_avg * 97 + 32  # read row + bucket + m x (matched row in, joined row out) + own-side delete / re-insert
                line["retract"] = {
                    "workload": "cfg3 retraction phase: auction U-/U+ pairs against the bid side held by the same operator "
                                f"({(W + K + V) * BATCH} bids stored), 2^19 pairs = 2^20 rows per step",
                    "metric": "input rows/s", "value": KR * 2 * RP / (rms / 1e3), "steps": KR, "ms_per_step": rms / KR,
                    "out_rows_per_input_row": m_avg,
                    "roofline": {"bound": "hbm", "kernel": "uni_hot_kernel<false,true,4> (inline-side rows: bucket + inline claim; chain walk + emit deferred to uni_tail_kernel)",
                                 "achieved": bpr * 2 * RP * rk_n / (rk_ms / 1e3) / 1e9 if rk_ms else None, "peak": peak, "unit": "GB/s",
                                 "frac": (bpr * 2 * RP * rk_n / (rk_ms / 1e3) / 1e9 / peak) if rk_ms else None,
                                 "algorithmic_bytes_per_row": bpr, "kernel_ms_avg": rk_ms / max(rk_n, 1), "traffic": None}}
                del ups_dev
            del join, batches_dev, chunks_dev
            torch.cuda.empty_cache()

        # ================================================================ leg: hot (SURVEY 8(d) cfg3 hot variant)
        if "hot" in legs and world == 1:
            KH, WH = min(K, 10), 3
            jh = new_join()
            build(jh, shuffle=False)
            hb = [gen_bids(BATCH, s * BATCH, SEED, N_BUILD, hot=True) for s in range(WH + KH + 1)]
            hdev = [dchunk(to_dev(b)) for b in hb]
            torch.cuda.synchronize()

            def run_hot(lo, hi, each=None):
                tot = 0
                for s2 in range(lo, hi):
                    device.join_push_device_async(jh, abi.SIDE_LEFT, hdev[s2], stream)
                    if s2 > lo:
                        o = device.join_collect(jh, stream)
                        tot += o.n_rows
                        if each:
                            each(o)
                o = device.join_collect(jh, stream)
                tot += o.n_rows
                if each:
                    each(o)
                return tot

            run_hot(0, WH)
            device.profile(jh, "join", True)
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record(stream)
            run_hot(WH, WH + KH)
            h1.record(stream)
            torch.cuda.synchronize()
            hms = h0.elapsed_time(h1)
            hk_ms, hk_n = device.profile(jh, "join", False)
            hcs = [0, 0]

            def add_hcs(o):
                a, b = o.checksum(CHECKSUM_WEIGHTS)
                hcs[0] += a
                hcs[1] = (hcs[1] + b) & ((1 << 64) - 1)

            run_hot(WH + KH, WH + KH + 1, add_hcs)
            hot_verify = (hcs[0], hcs[1], hb[WH + KH])
            hg = JOIN_BYTES_PER_ROW_STEP * BATCH * hk_n / (hk_ms / 1e3) / 1e9 if hk_ms else None
            line["hot"] = {"workload": "cfg3 hot variant: half of the bids go to 100 hot auctions (same-bucket atomics, long chains)",
                           "metric": "input rows/s", "value": KH * BATCH / (hms / 1e3), "steps": KH, "ms_per_step": hms / KH,
                           "roofline": {"bound": "hbm", "kernel": "uni_hot_kernel<false,false,4>", "achieved": hg, "peak": peak, "unit": "GB/s",
                                        "frac": hg / peak if hg else None, "algorithmic_bytes_per_row": JOIN_BYTES_PER_ROW_STEP,
                                        "kernel_ms_avg": hk_ms / max(hk_n, 1), "traffic": None}}
            del jh, hdev
            torch.cuda.empty_cache()

        # ================================================================ leg: e2e (host buffers, C ABI, COMPILED caller)
        def e2e_leg():
            """the same steps through the host-buffer entry point, driven by a compiled caller of the C ABI
            (tools/e2e_caller.cc, built by __graft_entry__.build()): pinned host StreamChunk buffers -> rwgpu_join_push ->
            EVERY output chunk view fetched and read -> release -- what the Rust shim does per message.  N>1: every rank
            runs its own caller on its own GPU and partition (as N independent shim instances would), started together."""
            exe = os.path.join(ROOT, "build", "e2e_caller")
            if not os.path.exists(exe):  # (a snapshot without build/: the caller only needs g++ and the library)
                if rank == 0:
                    sys.path.insert(0, ROOT)
                    import __graft_entry__
                    __graft_entry__.build_e2e_caller()
                if world > 1:
                    dist.barrier()
            if not os.path.exists(exe):
                raise RuntimeError("build/e2e_caller missing: run __graft_entry__.build()")
            env = dict(os.environ)
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            env["CUDA_VISIBLE_DEVICES"] = (vis.split(",")[local_rank] if vis else str(local_rank))
            torch.cuda.empty_cache()
            if world > 1:
                dist.barrier()  # the callers of all ranks start together
            def run_caller(mode):
                r = subprocess.run([exe, str(N_BUILD), str(BATCH), str(K), str(W), mode], capture_output=True, text=True, env=env, timeout=900)
                if r.returncode != 0:
                    raise RuntimeError(f"e2e_caller ({mode}) failed: {r.stderr[-500:]}")
                return json.loads(r.stdout.strip().splitlines()[-1])

            j = run_caller("async")
            js = run_caller("sync") if world == 1 else None
            al = int(j["output_columns_aliasing_input"])
            res = {"value": j["value"], "unit": "rows/s", "h2d_bytes_per_step": BATCH * (4 * 8 + 1),
                   "d2h_bytes_per_step": int(j["out_rows"]) * (8 * (8 - al) + 1) // K, "ffi_batch_rows": BATCH, "ms_per_step": j["ms_per_step"],
                   "output_columns_aliasing_input": al, "chunk_views_read_per_step": j["chunk_views_read_per_step"],
                   "verified": bool(j.get("verified")), "verification": {"rows": j.get("verify_rows"), "checksum": j.get("verify_checksum"),
                                                                          "how": "one more step after the timed ones, every output row read by the "
                                                                                 "caller and compared with the join evaluated on the host"},
                   "note": "compiled caller (tools/e2e_caller.cc) = what the executor shim does per message: pinned host StreamChunk buffers -> "
                           "rwgpu_join_push_async (step s+1 launched before step s is collected) -> rwgpu_join_collect_out -> every one of the "
                           "output chunk views fetched and read -> rwgpu_out_release; the bid-side output columns alias the caller's input "
                           "buffers (rwgpu.h), the rest is read back over PCIe"}
            if js is not None:
                res["one_call_at_a_time"] = {"value": js["value"], "ms_per_step": js["ms_per_step"], "verified": bool(js.get("verified")),
                                             "note": "the same caller through the synchronous rwgpu_join_push (H2D / kernels / D2H overlap inside a call only)"}
            return res

        if "e2e" in legs:
            res, ok = None, 1.0
            try:
                res = e2e_leg()
            except Exception as ex:  # (at N>1 every rank still reaches the collective below)
                print(f"[rank {rank}] e2e leg failed: {ex!r}", file=sys.stderr)
                ok = 0.0
            torch.cuda.empty_cache()
            if world > 1:
                t = torch.tensor([res["ms_per_step"] if res else 0.0, -ok], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)  # slowest rank; any failure makes the second entry 0
                if float(t[1].item()) < 0.0 and res:
                    res["ms_per_step"] = float(t[0].item())
                    res["value"] = world * BATCH / (res["ms_per_step"] / 1e3)
                    res["h2d_bytes_per_step"] *= world
                    res["d2h_bytes_per_step"] *= world
                    res["note"] += f"; N={world}: host input partitioned per rank, max over ranks"
                else:
                    res = None
            if res:
                line["e2e"] = res

        # ================================================================ leg: agg (secondary, configs[1]; SURVEY 8(d) cfg2 A / B / R)
        def agg_leg(variant):
            """variant A: uniform keys; B: half of the rows on 128 hot auctions; R: 10 % of the rows retract a row of the
            previous epoch (count / sum only: max is an append-only value state).  Every epoch's delta is compared with the CPU
            restatement through (row count, checksum) -- collected outside the timed loop on a second pass."""
            calls = ("(count:int8)", "(sum:int8 $1:int8)") + (() if variant == "R" else ("(max:int8 $1:int8)",))
            _, src = MockSource.channel()
            agg = HashAggExecutor(be, src.into_executor([abi.T_INT64] * 2, []), variant != "R",
                                  [AggCall.from_pretty(c) for c in calls], 0, [0], group_capacity_hint=2 * AGG_KEYS)
            n_ep_w, n_ep = 4, 60
            seed = {"A": AGG_SEED, "B": AGG_SEED + 1, "R": AGG_SEED + 2}[variant]
            ep_host, ep_dev = [], []
            prev = None
            for e in range(n_ep_w + n_ep):
                k, p = gen_agg_rows(AGG_EPOCH_ROWS, e * AGG_EPOCH_ROWS, seed, hot=(variant == "B"))
                ops = np.ones(AGG_EPOCH_ROWS, np.uint8)
                if variant == "R" and prev is not None:
                    nd = AGG_EPOCH_ROWS // 10  # rows 0, 10, 20, ... retract row i of the previous epoch (each at most once)
                    sel = np.arange(nd) * 10
                    live = prev[2][sel] == 1
                    k[sel[live]], p[sel[live]] = prev[0][sel[live]], prev[1][sel[live]]
                    ops[sel[live]] = 2
                prev = (k, p, ops)
                ep_host.append((ops, k, p))
                ep_dev.append(device.DeviceChunk(torch.from_numpy(ops).cuda(), [torch.from_numpy(k).cuda(), torch.from_numpy(p).cuda()],
                                                 [abi.T_INT64] * 2))
            torch.cuda.synchronize()
            for e in range(n_ep_w):
                device.agg_push_device(agg, ep_dev[e], stream)
                device.agg_flush_device(agg, e + 1, stream)
            device.profile(agg, "agg", True)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            # launch / collect split: barrier e is only ENQUEUED after its epoch's rows; its delta is collected while the
            # GPU already works on epoch e + 1 (two output sets), so the host never sits between two launches
            delta_rows = 0
            n_v = 6  # the last n_v epochs are checksummed (outside the timed loop: their deltas are kept by value)
            for e in range(n_ep_w, n_ep_w + n_ep):
                device.agg_push_device(agg, ep_dev[e], stream)
                device.agg_flush_device_async(agg, e + 1, stream)
                if e > n_ep_w:
                    delta_rows += device.agg_flush_collect(agg, stream).n_rows
            delta_rows += device.agg_flush_collect(agg, stream).n_rows
            a1.record(stream)
            torch.cuda.synchronize()
            ams = a0.elapsed_time(a1)
            akern_ms, akern_n = device.profile(agg, "agg", False)
            # verification epochs (untimed): n_v more epochs, each delta checksummed, against the CPU restatement fed everything
            vr = vc = 0
            v_host = []
            for e in range(n_ep_w + n_ep, n_ep_w + n_ep + n_v):
                k, p = gen_agg_rows(AGG_EPOCH_ROWS, e * AGG_EPOCH_ROWS, seed, hot=(variant == "B"))
                ops = np.ones(AGG_EPOCH_ROWS, np.uint8)
                v_host.append((ops, k, p))
                device.agg_push_device(agg, device.DeviceChunk(torch.from_numpy(ops).cuda(), [torch.from_numpy(k).cuda(), torch.from_numpy(p).cuda()],
                                                               [abi.T_INT64] * 2), stream)
                rows_v, cs_v = device.agg_flush_device(agg, e + 1, stream).checksum((1,) * (1 + len(calls)))
                vr += rows_v
                vc = (vc + cs_v) & ((1 << 64) - 1)
            fc = FastCpu().f
            fc.rwf_agg_checksum.restype = C.c_uint64
            fc.rwf_agg_checksum.argtypes = [C.c_void_p]
            ha = fc.rwf_agg_new(0 if variant == "R" else 1)
            fc.rwf_agg_reserve(ha, 2 * AGG_KEYS)
            want_rows = 0
            cs0 = 0
            for idx, (ops, k, p) in enumerate(ep_host + v_host):
                fc.rwf_agg_push(ha, len(ops), ops.ctypes.data, k.ctypes.data, p.ctypes.data)
                r = fc.rwf_agg_flush(ha)
                if idx == len(ep_host) - 1:
                    cs0 = fc.rwf_agg_checksum(ha)
                if idx >= len(ep_host):
                    want_rows += r
            want_cs = (fc.rwf_agg_checksum(ha) - cs0) & ((1 << 64) - 1)
            fc.rwf_agg_free(ha)
            d = delta_rows / (n_ep * AGG_EPOCH_ROWS)
            # SURVEY 8(d): B_agg = W_in + 1.125 + (K + 2A) + d_groups * (2 (K + A_out + 1) + K + A + A_out), d_groups = delta rows / 2
            A = 8 * len(calls)
            bpr = 16 + 1.125 + 8 + 2 * A + (d / 2) * (2 * (8 + A + 1) + 8 + A + A)
            agbs = AGG_BYTES_PER_ROW_FLOOR * AGG_EPOCH_ROWS * akern_n / (akern_ms / 1e3) / 1e9 if akern_ms else None
            step_gbs = bpr * n_ep * AGG_EPOCH_ROWS / (ams / 1e3) / 1e9
            return {
                "workload": f"nexmark_q4_hashagg_cfg2 variant {variant}: {', '.join(calls)} GROUP BY auction; 2^20 keys "
                            + {"A": "uniform", "B": "half of the rows on 128 hot keys", "R": "uniform, 10 % of the rows retract a row of the previous epoch"}[variant]
                            + "; 2^18-row epochs (256 chunks x 1024), barrier per epoch (launch / collect split)",
                "metric": "rows/s", "value": n_ep * AGG_EPOCH_ROWS / (ams / 1e3), "epochs": n_ep, "ms_per_epoch": ams / n_ep,
                "delta_rows_per_input_row": d,
                "verified": bool((vr, vc) == (want_rows, want_cs)),
                "verification": {"epochs": n_v, "gpu_delta_rows": vr, "cpu_delta_rows": want_rows, "gpu_checksum": f"{vc:016x}", "cpu_checksum": f"{want_cs:016x}"},
                "roofline": {"bound": "hbm", "kernel": f"agg_apply_fast_kernel<{len(calls)}>", "achieved": agbs, "peak": peak, "unit": "GB/s",
                             "frac": agbs / peak if agbs else None, "traffic": ncu_traffic("agg_apply_fast_kernel"), "peak_source": which,
                             "algorithmic_bytes_per_row": AGG_BYTES_PER_ROW_FLOOR, "kernel_ms_avg": akern_ms / max(akern_n, 1)},
                "epoch_roofline": {"what": "apply + barrier delta together (the whole epoch), bytes incl. the emitted delta rows",
                                   "algorithmic_bytes_per_row": bpr, "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak}}

        if "agg" in legs and world == 1:
            line["secondary"] = agg_leg("A")
            line["secondary_hot_keys"] = agg_leg("B")
            line["secondary_retract"] = agg_leg("R")
            torch.cuda.empty_cache()

        # ================================================================ leg: q1 (BASELINE configs[0], SURVEY 8(d) cfg1 plumbing)
        if "q1" in legs and world == 1:
            from risingwave_b200.executor import ProjectExecutor
            from risingwave_b200.stream_chunk import Column as HCol, StreamChunk as HChunk
            n1 = 1 << 20
            b1 = gen_bids(n1, 0, SEED, N_BUILD)  # (auction, date_time, bidder, price)
            cols_h = [b1[0], b1[2], b1[3], b1[1]]  # q1 order: auction, bidder, price, date_time
            _, s1 = MockSource.channel()
            expr = "(divide:int8 (multiply:int8 $2:int8 908:int8) 1000:int8)"
            pe = ProjectExecutor(be, s1.into_executor(T4, []), [expr])
            hchunk = HChunk(np.ones(n1, np.uint8), [HCol(abi.T_INT64, c) for c in cols_h])
            pe.apply_project_exprs(hchunk)
            t0 = time.perf_counter()
            reps = 5
            for _ in range(reps):
                out1 = pe.apply_project_exprs(hchunk)  # InputRef columns are passed through by pointer; one expression is computed
            host_s = (time.perf_counter() - t0) / reps
            dch = dchunk(to_dev(cols_h))
            q0, q1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            device.project_device(dch, pe._exprs, pe.schema, stream)
            q0.record(stream)
            for _ in range(20):
                dcols, dvalid, dnull = device.project_device(dch, pe._exprs, pe.schema, stream)
            q1e.record(stream)
            torch.cuda.synchronize()
            dev_ms = q0.elapsed_time(q1e) / 20
            want = (cols_h[2] * 908) // 1000  # prices are non-negative and small: no overflow, truncation == floor
            ok = bool(np.array_equal(out1.columns[0].data, want) and np.array_equal(dcols[0].cpu().numpy(), want) and int(dnull.sum().item()) == 0)
            pgbs = 17.0 * n1 / (dev_ms / 1e3) / 1e9  # 8 B read + 8 B + 1 B written per row
            line["q1"] = {"workload": "nexmark_q1_project_cfg1: one 2^20-row chunk, Project(auction, bidder, price * 908 / 1000, date_time)",
                          "metric": "rows/s", "value": n1 / (dev_ms / 1e3), "ms_per_chunk": dev_ms,
                          "e2e": {"value": n1 / host_s, "unit": "rows/s", "note": "rwgpu_project with a HOST chunk: upload, kernel, download"},
                          "verified": ok,
                          "roofline": {"bound": "hbm", "kernel": "project_kernel", "achieved": pgbs, "peak": peak, "unit": "GB/s", "frac": pgbs / peak,
                                       "algorithmic_bytes_per_row": 17.0, "kernel_ms_avg": dev_ms, "traffic": None}}

        # ================================================================ leg: generic (the path of the 7 non-inner join types)
        if "generic" in legs and world == 1:
            # LEFT OUTER bid x auction on the generic path (join_prepare_kernel -> cub scan + radix sort by (key group, row) ->
            # join_serial_kernel: one thread per join key runs hash_join_utils' match loop literally, degrees included).
            # 2^20 auctions resident; a step = 2^18 bids, 1/8 of them without a partner (NULL-padded output rows); then 2^18
            # auction inserts, half of which find waiting bids (each flips its NULL row: U-/U+ ... here Delete + Insert pairs).
            NG, BG, KG, WG = 1 << 20, 1 << 18, min(K, 8), 2
            _, gl = MockSource.channel()
            _, gr = MockSource.channel()
            jg = HashJoinExecutor(be, abi.JOIN_LEFT_OUTER, gl.into_executor(T4, [1]), gr.into_executor(T4, [0]),
                                  JoinParams([0], [1]), JoinParams([0], []), [False], capacity_hint=(NG, NG))
            ag = gen_auctions(NG, SEED + 77)
            device.join_push_device(jg, abi.SIDE_RIGHT, dchunk(to_dev(ag)), stream)
            gb = [gen_bids(BG, s * BG, SEED + 5, NG + NG // 8) for s in range(WG + KG)]  # ids >= NG have no auction yet
            gdev = [dchunk(to_dev(b)) for b in gb]
            torch.cuda.synchronize()
            for s in range(WG):
                device.join_push_device(jg, abi.SIDE_LEFT, gdev[s], stream)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0g = device.launches(jg, "join")
            g0.record(stream)
            g_rows = g_null = 0
            for s in range(WG, WG + KG):
                v = device.join_push_device(jg, abi.SIDE_LEFT, gdev[s], stream)
                g_rows += v.n_rows
            g1.record(stream)
            torch.cuda.synchronize()
            gms = g0.elapsed_time(g1)
            lg = device.launches(jg, "join") - l0g
            # verification of the last step on the host: every bid emits exactly one row; unmatched ones are NULL-padded
            vv = device.join_push_device(jg, abi.SIDE_LEFT, dchunk(to_dev(gen_bids(BG, (WG + KG) * BG, SEED + 5, NG + NG // 8))), stream)
            vb = gen_bids(BG, (WG + KG) * BG, SEED + 5, NG + NG // 8)
            pos_of = np.empty(NG, np.int64)
            pos_of[ag[0]] = np.arange(NG)
            matched = vb[0] < NG
            vis_v = vv.visible()  # (the generic path's output has invisible rows: it is not compacted)
            keep_v = None if vis_v is None else vis_v.cpu().numpy()
            got = [vv.column(k).cpu().numpy() for k in range(8)]
            if keep_v is not None:
                got = [g[keep_v] for g in got]
            ok = len(got[0]) == BG
            if ok:
                order_g = np.argsort(got[1], kind="stable")  # date_time is unique: aligns output rows with input rows
                order_w = np.argsort(vb[1], kind="stable")
                for k in range(4):
                    ok = ok and bool(np.array_equal(got[k][order_g], vb[k][order_w]))
                m_w = matched[order_w]
                for k in range(4):
                    want_k = ag[k][pos_of[np.where(m_w, vb[0][order_w], 0)]]
                    ok = ok and bool(np.array_equal(got[4 + k][order_g][m_w], want_k[m_w]))
                ok = ok and bool(vv.valid_ptrs[4])  # the unmatched rows carry NULLs on the auction side
            # the other direction: new auctions, half of which find waiting (NULL-padded) bids
            new_ids = NG + np.arange(0, NG // 8, dtype=np.int64)
            upd = [new_ids, new_ids % 1000, 10 + new_ids % 5, new_ids * 3]
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record(stream)
            vu = device.join_push_device(jg, abi.SIDE_RIGHT, dchunk(to_dev(upd)), stream)
            h1.record(stream)
            torch.cuda.synchronize()
            ums = h0.elapsed_time(h1)
            line["generic_join"] = {
                "workload": f"LEFT OUTER bid x auction, {NG} auctions resident, {BG} bids per step (1/9 without a partner: NULL-padded rows); "
                            f"then {NG // 8} new auctions whose waiting bids flip from NULL-padded to matched",
                "metric": "input rows/s", "value": KG * BG / (gms / 1e3), "steps": KG, "ms_per_step": gms / KG, "out_rows_per_step": g_rows / KG,
                "launches_per_step": lg / KG, "verified": bool(ok),
                "degree_flip_step": {"input_rows": int(NG // 8), "out_rows": int(vu.n_rows), "ms": ums, "rows_per_s": (NG // 8) / (ums / 1e3)},
                "note": "the generic path runs hash_join_utils' per-key match loop on ONE thread per join key (exact degree semantics); "
                        "its cost is the sort by key group, not HBM bandwidth: no roofline is claimed for it"}
            del jg, gdev
            torch.cuda.empty_cache()

        # ================================================================ leg: chain (join -> filter -> project -> agg in HBM)
        if "chain" in legs and world == 1:
            from risingwave_b200.executor import parse_filter_expr
            join3 = new_join()
            build(join3, shuffle=False)
            _, src3 = MockSource.channel()
            agg3 = HashAggExecutor(be, src3.into_executor([abi.T_INT64] * 2, []), True,
                                   [AggCall.from_pretty(c) for c in ("(count:int8)", "(max:int8 $1:int8)")], 0, [0],
                                   group_capacity_hint=2 * N_BUILD)
            # join output: bid (auction, date_time, bidder, price) | auction (id, seller, category, expires)
            expr = "(and:boolean (less_than_or_equal:boolean $2:int8 $5:int8) (greater_than_or_equal:boolean $3:int8 1048576:int8))"
            tp = parse_filter_expr(expr)
            terms = (abi.RwFilterTerm * len(tp))()
            for k, (cmp, lhs, rhs, const) in enumerate(tp):
                terms[k].cmp, terms[k].lhs_col, terms[k].rhs_col, terms[k].rhs_const = cmp, lhs, rhs, const
            KC, WC = min(K, 12), 3
            cdev = [dchunk(to_dev(b)) for b in batches_host[:KC + WC]]
            torch.cuda.synchronize()
            f0 = [torch.cuda.Event(enable_timing=True) for _ in range(KC + WC)]
            f1 = [torch.cuda.Event(enable_timing=True) for _ in range(KC + WC)]
            passed = deltas = 0

            def chain_step(s):
                nonlocal passed, deltas
                view = device.join_push_device(join3, abi.SIDE_LEFT, cdev[s], stream)
                raw = abi.RwChunk()
                cols = (abi.RwColumn * view.n_cols)()
                for k in range(view.n_cols):
                    cols[k].type, cols[k].data, cols[k].validity = view.col_types[k], view.col_ptrs[k], view.valid_ptrs[k]
                raw.n_rows, raw.n_cols, raw.ops, raw.visibility, raw.columns = view.n_rows, view.n_cols, view.ops_ptr, view.vis_ptr, cols
                f0[s].record(stream)
                f_ops, f_vis, f_n = device.filter_device(raw, view.n_rows, terms, False, stream)
                f1[s].record(stream)
                proj = abi.RwChunk()  # Project (auction, price): column pointers only
                pcols = (abi.RwColumn * 2)()
                for k, c in enumerate((0, 3)):
                    pcols[k].type, pcols[k].data, pcols[k].validity = view.col_types[c], view.col_ptrs[c], view.valid_ptrs[c]
                proj.n_rows, proj.n_cols, proj.ops, proj.visibility, proj.columns = view.n_rows, 2, f_ops.data_ptr(), f_vis.data_ptr(), pcols
                device._check(device._lib().rwgpu_agg_push_device(agg3._h, C.byref(proj), C.c_void_p(stream.cuda_stream)))
                deltas += device.agg_flush_device(agg3, s + 1, stream).n_rows  # a barrier after every 2^20-row batch
                passed += int(f_n.item())

            for s in range(WC):
                chain_step(s)
            passed = deltas = 0
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            for s in range(WC, WC + KC):
                chain_step(s)
            c1.record(stream)
            torch.cuda.synchronize()
            cms = c0.elapsed_time(c1)
            fms = sum(a.elapsed_time(b) for a, b in zip(f0[WC:], f1[WC:])) / KC
            FILTER_BYTES_PER_ROW = 3 * 8 + 1 + 1 + 0.125  # three predicate columns + ops read; ops + visibility written
            fgbs = FILTER_BYTES_PER_ROW * BATCH / (fms / 1e3) / 1e9
            line["chain"] = {
                "workload": "q4-shaped device-resident chain: bid JOIN auction -> Filter(bidder <= seller AND price >= 2^20) -> "
                            "Project(auction, price) -> HashAgg(count, max GROUP BY auction), a barrier per 2^20-row batch",
                "metric": "bid rows/s through the whole chain", "value": KC * BATCH / (cms / 1e3), "steps": KC, "ms_per_step": cms / KC,
                "filter_selectivity": passed / (KC * BATCH), "agg_delta_rows_per_step": deltas / KC,
                "filter_roofline": {"bound": "hbm", "kernel": "filter_kernel", "achieved": fgbs, "peak": peak, "unit": "GB/s",
                                    "frac": fgbs / peak, "algorithmic_bytes_per_row": FILTER_BYTES_PER_ROW, "kernel_ms_avg": fms,
                                    "traffic": None}}
            del join3, agg3, cdev
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    allowed, phys, quota = cpu_topology()
    if verify_gpu is not None:
        # the same V batches (all ranks' rows) against the same build side through the CPU restatement
        auct_all = [np.concatenate(c) for c in zip(*[gen_auctions(N_BUILD, SEED + r * 1000, r * N_BUILD) for r in range(world)])]
        vb = [[np.concatenate(c) for c in zip(*[gen_bids(BATCH, bid_start(r, K + W + v), SEED, N_BUILD * world) for r in range(world)])]
              for v in range(V)]
        ref = cpu_join_run(auct_all, vb, phys[:64], 0)
        ok = (ref["out_rows"], ref["checksum"]) == verify_gpu
        line["verified"] = bool(ok)
        line["verification"] = {"batches": V, "rows_per_batch": BATCH * world, "gpu_out_rows": verify_gpu[0], "cpu_out_rows": ref["out_rows"],
                                "gpu_checksum": f"{verify_gpu[1]:016x}", "cpu_checksum": f"{ref['checksum']:016x}",
                                "how": "after the timed region the same handle(s) take V more 2^20-row batches per GPU (through the exchange "
                                       "at N>1); row count and sum over output rows of sign(op) * sum_k w_k * col_k (mod 2^64) are compared "
                                       "with oracle/fastcpu.cc fed the same build side and batches"}
        if not ok:
            print("VERIFICATION FAILED: " + json.dumps(line["verification"]), file=sys.stderr)
    if retract_verify is not None:
        # CPU replay: build, every bid batch the handle received, the timed update steps, then the verification step
        rows_g, cs_g, warm_ups, ver_up = retract_verify
        ca = CpuActors(phys[:64])
        ca.reserve(auct)
        ca.run(1, [auct])
        ca.run(0, batches_host)
        ca.run(1, warm_ups)
        rv = ca.run(1, [ver_up])
        ca.close()
        want_rows, want_cs = rv["out_rows"], rv["checksum"]
        line["retract"]["verified"] = bool((rows_g, cs_g) == (want_rows, want_cs))
        line["retract"]["verification"] = {"gpu_out_rows": rows_g, "cpu_out_rows": want_rows, "gpu_checksum": f"{cs_g:016x}",
                                           "cpu_checksum": f"{want_cs:016x}"}
    if hot_verify is not None:
        rows_g, cs_g, vb_hot = hot_verify
        ref = cpu_join_run(gen_auctions(N_BUILD, SEED), [vb_hot], phys[:64], 0)
        line["hot"]["verified"] = bool((rows_g, cs_g) == (ref["out_rows"], ref["checksum"]))
        line["hot"]["verification"] = {"gpu_out_rows": rows_g, "cpu_out_rows": ref["out_rows"], "gpu_checksum": f"{cs_g:016x}",
                                       "cpu_checksum": f"{ref['checksum']:016x}"}
    if "cpu" in legs and world == 1:
        nb = 5
        sample = [gen_bids(1 << 20, s << 20, SEED, N_BUILD) for s in range(nb)]
        r1 = cpu_join_run(gen_auctions(N_BUILD, SEED), sample, phys[:1], 1)
        line["cpu_baseline"] = {"value": r1["value"], "unit": "rows/s", "cores": 1, "kind": "port",
                                "sample": f"oracle/fastcpu.cc single actor pinned to one core, 10M-row build (untimed) then {nb - 1} x 2^20 bid "
                                          f"rows in 1024-row chunks ({r1['wall_s']:.1f} s); host: {len(allowed)} logical / {len(phys)} physical "
                                          f"cores allowed, cgroup quota {quota}"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """CPU arm: restatement of the reference algorithm (oracle/fastcpu.cc) on the host cores, rank 0 only.
    One single-threaded actor per core as the reference deploys them (actor.rs:209-232,272); the actor count is
    chosen by measurement (one per physical core / one per logical CPU / the cgroup quota) and the parallel
    efficiency against a single pinned actor is printed with the line."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    allowed, phys, quota = cpu_topology()
    K, W = args.steps, args.warmup
    n_steps = min(K, 64)  # the same number of 2^20-row steps as the GPU arm: the left-side state (rows per key) grows alike
    auct = gen_auctions(N_BUILD, SEED)
    batches = [gen_bids(BATCH, s * BATCH, SEED, N_BUILD) for s in range(W + n_steps)]
    one = cpu_join_run(auct, batches, phys[:1], W)
    cands = {len(phys): phys}
    if len(allowed) > len(phys):
        cands[len(allowed)] = allowed
    if quota and 1 <= int(quota) < len(phys):
        cands[int(quota)] = phys[:int(quota)]
    if len(phys) >= 16:
        cands[len(phys) // 2] = phys[::2]
    sweep = []
    for P in sorted(cands):
        r = cpu_join_run(auct, batches, cands[P], W)
        r["efficiency_vs_one_actor"] = r["value"] / (P * one["value"]) if one["value"] else None
        sweep.append(r)
        print(f"[cpu arm] P={P}: {r['value'] / 1e6:.1f} M rows/s, wall {r['wall_s']:.3f} s, busy min/mean/max "
              f"{r['busy_s_min']:.3f}/{r['busy_s_mean']:.3f}/{r['busy_s_max']:.3f} s, pin failures {r['pin_failures']}, "
              f"efficiency {r['efficiency_vs_one_actor']:.2f}", file=sys.stderr)
    best = max(sweep, key=lambda r: r["value"])
    v, P = best["value"], best["actors"]
    line = {"impl": "reference", "metric": "Nexmark q7/q8-shaped streaming HashJoin input rows/s", "value": v, "unit": "rows/s",
            "n_gpus": world, "steps": n_steps, "warmup": W, "ms_per_step": best["wall_s"] / n_steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": bench_config(1),
            "cpu_baseline": {"value": v, "unit": "rows/s", "cores": P, "kind": "port",
                             "sample": f"oracle/fastcpu.cc: {P} single-threaded actors pinned one per core (vnode-partitioned input, tables "
                                       f"first-touched on the actor's thread, no per-step rendezvous), 10M-row build untimed, {n_steps} steps "
                                       f"of 2^20 bid rows in 1024-row chunks; the Rust reference cannot be built here"},
            "cpu_arm": {"allowed_logical_cpus": len(allowed), "physical_cores": len(phys), "cgroup_cpu_quota": quota,
                        "one_actor_rows_per_s": one["value"], "sweep": sweep,
                        "parallel_efficiency": best["efficiency_vs_one_actor"]},
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--legs", default="value,retract,hot,e2e,agg,q1,chain,generic,cpu",
                    help="comma list of: value,retract,hot,e2e,agg,q1,chain,generic,cpu (subset for ncu runs; retract needs value)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the join output of the last timed step of the value leg (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or "value" not in args.legs.split(",")):
        ap.error("--dump-outputs needs --impl ours and the value leg")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    # stdout carries exactly ONE line (the JSON): everything a library prints there on its own (NCCL's "NCCL version ..."
    # banner at communicator creation, for one) is sent to stderr for the duration of the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = io.StringIO()
    try:
        with contextlib.redirect_stdout(out):
            if args.impl == "reference":
                run_reference(args)
            else:
                run_ours(args)
    finally:
        sys.stdout.flush()
        try:
            C.CDLL(None).fflush(None)  # C stdio buffers too (NCCL printf()s its banner: it would surface at exit)
        except Exception:
            pass
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    lines = [ln for ln in out.getvalue().splitlines() if ln.strip()]
    json_lines = [ln for ln in lines if ln.lstrip().startswith("{")]
    for ln in lines:
        if ln not in json_lines:
            print(ln, file=sys.stderr)
    if json_lines:
        print(json_lines[-1], flush=True)


if __name__ == "__main__":
    main()
