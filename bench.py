#!/usr/bin/env python
"""bench.py -- measurement of the batched edit-distance hot path (BASELINE.json metric: GCUPS and alignments/s).

Headline workload at N GPUs (weak scaling): BASELINE.json configs[1] per GPU -- 1,000,000 x 150 bp DNA reads
(3 % sub/ins/del, seeded: edlib_b200/workloads.py) aligned HW (infix), EDLIB_TASK_DISTANCE, k = -1, to ONE shared
target: the E. coli DH1 genome of the reference's test data (4,630,707 bp; `--target synthetic` = uniform-random
5,000,000 bp instead, also reported as a second record).  One "step" = one pass of the hot path over the batch.

  value   nominal GCUPS = sum(queryLength * targetLength) / time / 1e9 over all ranks (SURVEY.md 8d: the same formula
          for CPU and GPU whatever either of them skips), batch already resident in HBM (edlibB200BatchCompute: seed
          index of the target, every kernel, results back on the host), barrier + synchronize, max over ranks.
  e2e     the same metric through the reference-facing call edlibAlignBatch() with HOST buffers (pack + H2D +
          kernels + D2H + one malloc'd array per result inside the timed region).
  roofline  per-kernel CUDA-event times of a step (`kernels_ms`); for the DOMINANT kernel its algorithmic bytes per
          launch / its device time against the measured HBM peak (MEASURED_PEAKS.json), its DRAM traffic from the
          committed ncu launch list (profiles/step_traffic.json) and -- the bound that matters for bit-vector work --
          its integer-issue fraction (`int_issue_frac`: logic-pipe instructions the recurrences need / time / peak).
  cpu_baseline  the reference build (oracle/_ref) on this box's host cores, bounded sample, results compared.

Sub-records (N = 1, skipped with --no-extras): `synthetic_target`, `sensitivity` (1 % unrelated reads / 8 % error /
repeat-rich target), `config3` (100k x 10 kbp NW k=500 LOC), `config4` (1M x 150 bp HW PATH + CIGAR), each with
end-to-end time, kernel time, its own roofline, a CPU sample and full-field parity on that sample; `sweep_kernel`
(the full-width Myers kernel alone).  `strong` (every N): BASELINE configs[4] -- 10M reads (seed 44) sharded over the
ranks, NCCL broadcast of the target and gather of the distances INSIDE the timed step.

`--impl reference` times the reference's own CPU implementation instead (same metric and config).
Multi-GPU: launched by torchrun, one rank per GPU.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

from edlib_b200 import sharding, workloads  # noqa: E402
from edlib_b200._ffi import AlignConfig, AlignResult, EdlibLib, make_config, product_path  # noqa: E402

READ_LEN = 150
SYNTH_TARGET_LEN = 5_000_000
MODE_NW, MODE_HW = 0, 2
TASK_DISTANCE, TASK_LOC, TASK_PATH = 0, 1, 2


class Stats(C.Structure):  # include/edlib_b200.h EdlibB200Stats
    _fields_ = [("kernelMs", C.c_double), ("k1Ms", C.c_double), ("launches", C.c_int), ("filterWindows", C.c_int),
                ("h2dBytes", C.c_longlong), ("d2hBytes", C.c_longlong), ("k1Cells", C.c_longlong),
                ("wCells", C.c_longlong), ("filterDecided", C.c_longlong), ("filterFallback", C.c_longlong)]


RESULT_DTYPE = np.dtype([("status", "<i4"), ("editDistance", "<i4"), ("endLocations", "<u8"), ("startLocations", "<u8"),
                         ("numLocations", "<i4"), ("pad0", "<i4"), ("alignment", "<u8"), ("alignmentLength", "<i4"),
                         ("alphabetLength", "<i4")])
assert RESULT_DTYPE.itemsize == 48


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region: ONE nvidia-smi process (rank 0) watches
    the GPUs of all local ranks (a poller per rank would only add driver traffic)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_indices):
        self.rows, self.proc, self.idx = [], None, list(gpu_indices)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(str(i) for i in self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        """{gpu index: {"sm_mhz": median under load, "sm_max_mhz", "reasons", "samples"}}"""
        if not self.proc:
            return {}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        out = {}
        for gpu in self.idx:
            sm, mx, reasons = [], [], set()
            for r in self.rows:
                try:
                    if int(r[0]) != gpu:
                        continue
                    sm.append(float(r[1]))
                    mx.append(float(r[2]))
                except Exception:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            if sm:
                out[gpu] = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def effective_cores():
    """Host cores this process may really use: CPU affinity, bounded by a cgroup CPU quota when there is one
    (containers often show every hardware thread but grant far fewer)."""
    try:
        cores = float(len(os.sched_getaffinity(0)))
    except Exception:
        cores = float(os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2: "<quota|max> <period>"
            quota, period = f.read().split()[:2]
            if quota != "max" and float(period) > 0:
                cores = min(cores, max(1.0, float(quota) / float(period)))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read().strip())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                pr = float(f.read().strip())
            if q > 0 and pr > 0:
                cores = min(cores, max(1.0, q / pr))
        except Exception:
            pass
    return max(1, int(cores + 0.5))


def measured_traffic(n_reads, kernel):
    """DRAM bytes per step of a kernel from the committed ncu launch list (same batch size only)."""
    path = os.path.join(REPO, "profiles", "step_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        if int(t["reads"]) == int(n_reads) and kernel in t["kernels"]:
            k = t["kernels"][kernel]
            return (float(k["dram_bytes_read"]) + float(k["dram_bytes_write"])) / max(1, int(k.get("launches", 1)))
    except Exception:
        pass
    return None


# B200 integer issue peak for the half-rate logic pipe (profiles/r01_pipe_microbench.txt: LOP3/SHF 0.49
# warp-instructions/clk/SMSP): 148 SMs x 4 SMSPs x 32 lanes x 0.49 x SM clock
def int_issue_peak(sm_mhz):
    return 148 * 4 * 32 * 0.49 * sm_mhz * 1e6


def pointer_arrays(reads, target):
    n = reads.shape[0]
    qptr = (reads.ctypes.data + np.arange(n, dtype=np.uint64) * np.uint64(reads.shape[1])).astype(np.uint64)
    qlen = np.full(n, reads.shape[1], dtype=np.int32)
    tptr = np.full(n, target.ctypes.data, dtype=np.uint64)
    tlen = np.full(n, target.shape[0], dtype=np.int32)
    return qptr, qlen, tptr, tlen


def as_pp(a):
    return a.ctypes.data_as(C.POINTER(C.c_char_p))


def as_pi(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def ref_lib():
    ref_so = os.path.join(REPO, "oracle", "_ref", "libedlib_ref.so")
    if os.path.exists(ref_so):
        return EdlibLib(ref_so, prefix="edlib"), "reference"
    return EdlibLib(os.path.join(REPO, "oracle", "liboracle.so"), prefix="oracle"), "port"


def cpu_sample(pairs, mode, task, k, seconds_goal, threads, cells_of, want_cigar=False):
    """Times the reference build's edlibAlign on the first S of `pairs` (callable i -> (query bytes, target bytes)) with
    one Python thread per host core (ctypes releases the GIL during the call).  Returns every result field of the
    sample for the parity check."""
    from concurrent.futures import ThreadPoolExecutor
    from edlib_b200._ffi import result_to_dict
    lib, kind = ref_lib()
    cfg, _ = make_config(k, mode, task)
    total = pairs["n"]

    def one(i):
        q, t = pairs["get"](i)
        r = lib.align_raw(q, t, cfg)
        d = result_to_dict(r)
        if want_cigar and d.get("alignment") is not None:
            d["cigar"] = lib.cigar(d["alignment"])
        if r.status == 0:
            lib.free(r)
        return d

    with ThreadPoolExecutor(threads) as ex:
        t0 = time.time()
        list(ex.map(one, range(min(threads, total))))  # calibration: one alignment per thread
        per = max(time.time() - t0, 1e-3)
        sample = int(min(total, max(threads, seconds_goal / per * threads)))
        t0 = time.time()
        res = list(ex.map(one, range(sample)))
        wall = time.time() - t0
    cells = float(sum(cells_of(i) for i in range(sample)))
    return {"gcups": cells / wall / 1e9, "alignments_per_s": sample / wall, "sample": sample, "wall": wall, "kind": kind,
            "results": res}


def gpu_result_dict(res, i, with_alignment=False):
    """Every field of results[i] (numpy RESULT_DTYPE) as the dict _ffi.result_to_dict builds."""
    r = res[i]
    n = int(r["numLocations"])
    d = {"status": int(r["status"]), "editDistance": int(r["editDistance"]), "numLocations": n,
         "alignmentLength": int(r["alignmentLength"]), "alphabetLength": int(r["alphabetLength"])}
    d["endLocations"] = list(np.frombuffer(C.string_at(int(r["endLocations"]), 4 * n), dtype=np.int32)) if r["endLocations"] else None
    d["startLocations"] = list(np.frombuffer(C.string_at(int(r["startLocations"]), 4 * n), dtype=np.int32)) if r["startLocations"] else None
    d["alignment"] = C.string_at(int(r["alignment"]), int(r["alignmentLength"])) if r["alignment"] else None
    return d


def check_sample(res, ref_results, what, cigars=None):
    """Full-field parity of the CPU sample: status, editDistance, numLocations, endLocations[], startLocations[]
    (NULL-ness included), alignment bytes, alphabetLength (and the CIGAR string when given)."""
    for i, exp in enumerate(ref_results):
        got = gpu_result_dict(res, i)
        exp = dict(exp)
        cg = exp.pop("cigar", None)
        assert got == exp, "%s: result %d differs from the reference: %s vs %s" % (what, i, str(got)[:300], str(exp)[:300])
        if cigars is not None and cg is not None:
            assert cigars[i] == cg, "%s: CIGAR %d differs" % (what, i)
    return len(ref_results)


class Engine:
    """The product library through its C ABI (ctypes)."""

    def __init__(self, local_rank):
        self.lib = EdlibLib(product_path(), has_batch=True)
        L = self.L = self.lib.lib
        L.edlibB200SetDevice.argtypes = [C.c_int]
        assert L.edlibB200SetDevice(local_rank) == 0
        assert L.edlibB200Available() == 1, "CUDA path unavailable"
        L.edlibB200BatchPrepare.restype = C.c_void_p
        L.edlibB200BatchPrepare.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_int),
                                            C.c_int, AlignConfig]
        L.edlibB200BatchCompute.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.edlibB200BatchResults.argtypes = [C.c_void_p, C.c_void_p]
        L.edlibB200BatchFree.argtypes = [C.c_void_p]
        L.edlibB200FreeResults.argtypes = [C.c_void_p, C.c_int]
        L.edlibB200LastStats.argtypes = [C.POINTER(Stats)]
        L.edlibB200LastError.restype = C.c_char_p
        L.edlibB200LastKernelReport.argtypes = [C.c_char_p, C.c_int]
        L.edlibB200AlignmentsToCigar.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.edlibB200FreeCigars.argtypes = [C.c_void_p, C.c_int]
        L.edlibB200TargetPrepare.restype = C.c_void_p
        L.edlibB200TargetPrepare.argtypes = [C.c_void_p, C.c_int]
        L.edlibB200TargetFree.argtypes = [C.c_void_p]
        self.numa_node = int(L.edlibB200DeviceNumaNode())
        self.allocator_tuned = L.edlibB200TuneHostAllocator() == 0  # keep freed result arrays in the allocator (edlib_b200.h)
        self.libc = C.CDLL(None)
        self.libc.free.argtypes = [C.c_void_p]

    def kernel_report(self):
        buf = C.create_string_buffer(8192)
        self.L.edlibB200LastKernelReport(buf, 8192)
        out = {}
        for item in buf.value.decode().split(";"):
            if item:
                name, ms, cnt = item.split(":")
                out[name] = (float(ms), int(cnt))
        return out

    def align_batch(self, ptrs, n, cfg, res):
        qptr, qlen, tptr, tlen = ptrs
        rc = self.L.edlibAlignBatch(as_pp(qptr), as_pi(qlen), as_pp(tptr), as_pi(tlen), n, cfg,
                                    C.cast(res.ctypes.data, C.POINTER(AlignResult)))
        assert rc == 0, self.L.edlibB200LastError()

    def free(self, res):
        self.L.edlibB200FreeResults(res.ctypes.data, len(res))

    def cigars(self, res):
        n = len(res)
        out = (C.c_void_p * n)()
        assert self.L.edlibB200AlignmentsToCigar(res.ctypes.data, n, 1, out) == 0
        return out

    def free_cigars(self, cg):
        self.L.edlibB200FreeCigars(cg, len(cg))


def resident_steps(E, ptrs, n, cfg, steps, warmup, flush, barrier):
    """value leg: the batch resident in HBM, `steps` timed computes.  Returns timing, per-kernel times, results."""
    L = E.L
    qptr, qlen, tptr, tlen = ptrs
    batch = L.edlibB200BatchPrepare(as_pp(qptr), as_pi(qlen), as_pp(tptr), as_pi(tlen), n, cfg)
    assert batch, L.edlibB200LastError()
    st = Stats()
    for _ in range(warmup):
        flush()
        assert L.edlibB200BatchCompute(batch, C.byref(st)) == 0, L.edlibB200LastError()
    barrier()
    import torch
    kernel_ms, launches, step_s, per_kernel, filt = [], 0, [], {}, (0, 0, 0)
    for _ in range(steps):
        flush()
        t0 = time.perf_counter()
        assert L.edlibB200BatchCompute(batch, C.byref(st)) == 0, L.edlibB200LastError()
        torch.cuda.synchronize()
        step_s.append(time.perf_counter() - t0)
        kernel_ms.append(st.kernelMs)
        launches += st.launches
        filt = (int(st.filterDecided), int(st.filterFallback), int(st.filterWindows))
        for name, (ms, cnt) in E.kernel_report().items():
            a = per_kernel.setdefault(name, [0.0, 0])
            a[0] += ms / steps
            a[1] += cnt
    barrier()
    res = np.zeros(n, dtype=RESULT_DTYPE)
    assert L.edlibB200BatchResults(batch, res.ctypes.data) == 0
    assert (res["status"] == 0).all()
    L.edlibB200BatchFree(batch)
    kernels_ms = {k: round(v[0], 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1][0])}
    return {"step_s": step_s, "kernel_ms": float(np.mean(kernel_ms)) if kernel_ms else 0.0, "launches": launches,
            "kernels_ms": kernels_ms, "kernel_launches": {k: v[1] // max(steps, 1) for k, v in per_kernel.items()},
            "filter": {"decided": filt[0], "fallback": filt[1], "windows": filt[2]}, "res": res}


def e2e_steps(E, ptrs, n, cfg, steps, barrier, expect_ed=None, keep_last=False):
    """e2e leg: edlibAlignBatch with host buffers, one untimed warm-up, `steps` timed calls."""
    import torch
    times, h2d, d2h, last = [], 0, 0, None
    st = Stats()
    for it in range((1 + steps) if steps > 0 else 0):
        res = np.empty(n, dtype=RESULT_DTYPE)
        res.view(np.uint8).fill(0)  # the caller's result array exists (pages touched) before the call
        barrier()
        t0 = time.perf_counter()
        E.align_batch(ptrs, n, cfg, res)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if expect_ed is not None:
            assert (res["editDistance"] == expect_ed).all()
        E.L.edlibB200LastStats(C.byref(st))
        h2d, d2h = int(st.h2dBytes), int(st.d2hBytes)
        if keep_last and it == steps:
            last = res
        else:
            E.free(res)
        if it > 0:
            times.append(dt)
    return {"times": times, "h2d": h2d, "d2h": d2h, "res": last, "kernel_ms": float(st.kernelMs)}


def reads_roofline(rs, n_reads, target_len, nloc_sum, sm_mhz, peak, peak_src):
    """roofline block of a reads-vs-one-target step from its per-kernel times."""
    kernels_ms = rs["kernels_ms"]
    dominant = next(iter(kernels_ms)) if kernels_ms else None
    dom_s = kernels_ms.get(dominant, 0.0) / 1000.0 if dominant else 0.0
    dom_launches = max(1, rs["kernel_launches"].get(dominant, 1)) if dominant else 1
    bytes_alg = float(n_reads) * (READ_LEN + target_len + 8) + 4.0 * nloc_sum      # SURVEY.md 8d accounting
    bytes_unique = float(n_reads) * (READ_LEN + 8) + target_len + 4.0 * nloc_sum   # what any implementation must move
    kern = rs["kernel_ms"] / 1000.0
    windows = float(rs["filter"]["windows"])
    int_frac = None
    if dominant == "k1w":
        # unit = one window sweep: the read (150 B), its target window (lead-in m + t plus >= 2t+1 tracked columns:
        # 181 for t = 10), a 20-byte job and a 64-byte record
        unit, dom_units, dom_what = READ_LEN + 181 + 20 + 64, windows, "window sweeps x (read + target window + job + record)"
        # banded sweep (eb_core.h k1b_sweep): per column 14 LOP3 + 4 funnel shifts that the recurrences need on two words
        int_frac = windows * 181 * 18 / dom_s / int_issue_peak(sm_mhz) if dom_s > 0 else None
    elif dominant in ("k1", "k1_prefix"):
        unit = READ_LEN + target_len + 8
        dom_units = float(rs["filter"]["fallback"]) if dominant == "k1" else float(n_reads)
        dom_what = "whole-target sweeps x (read + target + result)"
        int_frac = dom_units * target_len * 5 * 7 / dom_s / int_issue_peak(sm_mhz) if dom_s > 0 else None
    elif dominant == "seed_plan":
        unit, dom_units = READ_LEN + 11 * (8 + 4 + 16) + 16, float(n_reads)
        dom_what = "reads x (read + 11 seeds x (bucket bounds + position + target symbols) + plan record)"
    else:
        unit, dom_units, dom_what = bytes_unique, 1.0, "bytes that must move in a step (reads + target + results)"
    dom_bytes = dom_units * unit / dom_launches
    dom_launch_s = dom_s / dom_launches
    achieved = dom_bytes / dom_launch_s / 1e9 if dom_launch_s > 0 else 0.0
    traffic = measured_traffic(n_reads, dominant)
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "kernel": dominant, "kernel_ms": dom_launch_s * 1000.0,
            "launches_per_step": dom_launches, "units": dom_units / dom_launches, "bytes_per_unit": unit,
            "bytes_algorithmic": dom_bytes, "units_are": dom_what, "int_issue_frac": int_frac,
            "kernels_ms": kernels_ms, "all_kernels_ms": kern * 1000.0,
            "step_unique_bytes": bytes_unique, "step_unique_frac": bytes_unique / kern / 1e9 / peak if kern > 0 else None,
            "step_nominal_bytes": bytes_alg,
            "note": "dominant kernel of the step by CUDA-event time, per launch.  The path is integer-issue bound (ncu: "
                    "profiles/), so the HBM fraction is low by construction; int_issue_frac counts the logic-pipe "
                    "instructions the recurrences need against the measured half-rate pipe peak.  step_unique_* = bytes that "
                    "must move (reads + target + results) over the device time of all kernels; step_nominal_bytes is SURVEY.md "
                    "8d's accounting (every alignment 'consumes' its whole target), which the exact seed filter does not execute"}


def dump_outputs(res, out_dir, prefix="", budget=63 << 20):
    """Writes what the caller of the timed path received from its last step, one .npy per field: edit_distance and
    num_locations (float32, one per read), end_locations and start_locations (float64, every location of every read in
    read order; start_locations only where the task returns them).  Past `budget` bytes of data (under 64 MB with the
    file headers), the reads are a fixed seeded sample, listed in sample_index.npy."""
    n = len(res)
    rows = np.arange(n)
    order = np.random.Generator(np.random.PCG64(0)).permutation(n)
    while True:
        nloc = res["numLocations"][rows].astype(np.int64)
        starts = bool(res["startLocations"][rows].any())
        size = len(rows) * (8 + (8 if len(rows) < n else 0)) + int(nloc.sum()) * (16 if starts else 8)
        if size <= budget or len(rows) <= 1:
            break
        rows = np.sort(order[:len(rows) // 2])

    def locations(field):
        out = np.empty(int(nloc.sum()), dtype=np.float64)
        at = 0
        for i, c in zip(rows, nloc):
            if c:
                out[at:at + c] = np.frombuffer(C.string_at(int(res[field][i]), 4 * int(c)), dtype=np.int32)
                at += c
        return out

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"edit_distance": res["editDistance"][rows].astype(np.float32),
              "num_locations": nloc.astype(np.float32), "end_locations": locations("endLocations")}
    if starts:
        arrays["start_locations"] = locations("startLocations")
    if len(rows) < n:
        arrays["sample_index"] = rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def run_reads_workload(E, target, reads, steps, warmup, e2e_n, flush, barrier, want_cpu=None, cpu_seconds=15.0, dump=None):
    """One reads-vs-one-target HW distance workload: resident value, e2e, optional CPU sample with parity.  `dump`:
    (directory, file prefix) for the results of the last timed step (dump_outputs)."""
    n = reads.shape[0]
    ptrs = pointer_arrays(reads, target)
    cfg, _ = make_config(-1, MODE_HW, TASK_DISTANCE)
    rs = resident_steps(E, ptrs, n, cfg, steps, warmup, flush, barrier)
    res = rs.pop("res")
    if dump:
        dump_outputs(res, *dump)
    eds = res["editDistance"].copy()
    nloc = res["numLocations"].copy()
    cpu = None
    if want_cpu:
        tb = target.tobytes()
        cs = cpu_sample({"n": n, "get": lambda i: (reads[i].tobytes(), tb)}, MODE_HW, TASK_DISTANCE, -1, cpu_seconds, want_cpu,
                        lambda i: READ_LEN * len(target))
        checked = check_sample(res, cs["results"], "config 2")
        cpu = {"value": cs["gcups"], "unit": "GCUPS", "cores": want_cpu, "gcups_per_core": cs["gcups"] / want_cpu,
               "alignments_per_s": cs["alignments_per_s"], "kind": cs["kind"],
               "sample": "first %d reads of the batch, %.1f s wall; every result field bit-exact vs the GPU" % (checked, cs["wall"])}
    E.free(res)
    ee = e2e_steps(E, ptrs, n, cfg, e2e_n, barrier, expect_ed=eds)
    return rs, ee, eds, nloc, cpu


def sweep_kernel_sample(reads=32768):
    """The full-width Myers sweep alone: this script in a child process with every filter stage off."""
    env = dict(os.environ, EDLIB_B200_FILTER_SEED_K="0", EDLIB_B200_FILTER_K1="0", EDLIB_B200_FILTER_K0="0")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--reads", str(reads), "--steps", "1", "--warmup", "1",
                              "--e2e-steps", "0", "--no-cpu-baseline", "--no-extras", "--target", "synthetic"], env=env,
                             capture_output=True, text=True, timeout=600)
        j = json.loads(out.stdout.strip().splitlines()[-1])
        k1 = j["roofline"]["kernels_ms"]["k1"]
        cells = float(reads) * READ_LEN * SYNTH_TARGET_LEN
        sm = (j.get("clocks") or {}).get("sm_mhz") or 1965.0
        # 5 x 32-bit words per column, 7 logic + 3 add instructions per word and column (eb_core.h: k1_step)
        logic_ops = float(reads) * SYNTH_TARGET_LEN * 5 * 7
        return {"kernel": "k1_kernel<5,HW> (150-row reads, every cell of every column)", "reads": reads, "kernel_ms": k1,
                "gcups": cells / (k1 / 1e3) / 1e9, "logic_lane_ops_per_s": logic_ops / (k1 / 1e3),
                "int_issue_frac": logic_ops / (k1 / 1e3) / int_issue_peak(sm),
                "note": "true cell updates per second of the DP kernel; int_issue_frac counts only the 7 LOP3 per word-column "
                        "that no formulation avoids, against the half-rate logic pipe peak"}
    except Exception as e:  # the sample is informative only
        return {"error": repr(e)[:200]}


def sensitivity(E, genome, base_reads, flush, barrier):
    """The headline batch under less friendly inputs (resident compute, 2 timed steps each): what the exact filter
    costs when reads do not map, carry more errors, or come from a repeat-rich target."""
    out = {}
    n = base_reads.shape[0]
    cfg, _ = make_config(-1, MODE_HW, TASK_DISTANCE)

    def run(target, reads, label, note):
        rs = resident_steps(E, pointer_arrays(reads, target), reads.shape[0], cfg, 2, 1, flush, barrier)
        res = rs.pop("res")
        ms = 1000.0 * float(np.mean(rs["step_s"]))
        out[label] = {"note": note, "ms_per_step": ms, "kernel_ms_per_step": rs["kernel_ms"],
                      "gcups": float(reads.shape[0]) * READ_LEN * len(target) / (ms / 1e3) / 1e9,
                      "filter": rs["filter"], "kernels_ms": rs["kernels_ms"],
                      "mean_edit_distance": float(res["editDistance"].mean()), "mean_num_locations": float(res["numLocations"].mean())}
        E.free(res)

    # (a) 1 % of the reads replaced by unrelated (uniform random) ones: no seed can decide them, they take the plain sweep
    reads = base_reads.copy()
    k = n // 100
    reads[:k] = workloads.random_dna(k * READ_LEN, 777).reshape(k, READ_LEN)
    run(genome, reads, "unrelated_1pct", "1 % of the reads are uniform-random 150-mers (no alignment below ~55 edits): every stage "
                                         "of the filter passes them on and they take the full-width sweep")
    # (b) 8 % per-base error instead of 3 %
    run(genome, workloads.reads_of(genome, n, READ_LEN, seed=42, rate=0.08), "error_8pct",
        "reads with 8 % sub/ins/del (mean distance ~11): more reads need the shorter-seed levels")
    # (c) repeat-rich target: 1 Mbp of unique sequence + 100 mutated (1 %) copies of a 3 kbp element + 2.1 kbp of a 7-mer tandem
    # (a long tandem stretch would make the OUTPUT explode: every period is an end location of every read inside it)
    uniq = workloads.random_dna(1_000_000, 5)
    elem = workloads.random_dna(3000, 6)
    buf = np.empty(8000, dtype=np.uint8)
    parts, at = [], 0
    for c in range(100):
        nxt = (c + 1) * 10_000
        parts.append(uniq[at:nxt])
        at = nxt
        m = workloads._synth().synth_mutate(elem.ctypes.data, len(elem), buf.ctypes.data, 0.01, 1000 + c)
        parts.append(buf[:m].copy())
    parts.append(uniq[at:])
    parts.append(np.tile(np.frombuffer(b"ACGGTCA", dtype=np.uint8), 2_100 // 7))
    rep = np.ascontiguousarray(np.concatenate(parts))
    run(rep, workloads.reads_of(rep, n, READ_LEN, seed=42, rate=0.03), "repeat_rich_target",
        "%d bp target: 1 Mbp unique + 100 diverged copies of a 3 kbp element (23 %% of the target) + a 2.1 kbp tandem repeat; "
        "reads drawn uniformly from it" % len(rep))
    return out


def config3(E, genome, pairs, steps, cores, cpu_seconds, peak, peak_src, barrier):
    """BASELINE configs[2]: `pairs` x 10 kbp queries vs their 3 %-mutated copies, NW, k = 500, EDLIB_TASK_LOC."""
    t0 = time.time()
    qbuf, tbuf, tlens = workloads.long_pairs_packed(genome, pairs, 10_000, seed=43, pinned=True, numa_node=E.numa_node)
    gen_s = time.time() - t0
    n = pairs
    qptr = (qbuf.ctypes.data + np.arange(n, dtype=np.uint64) * np.uint64(qbuf.shape[1])).astype(np.uint64)
    tptr = (tbuf.ctypes.data + np.arange(n, dtype=np.uint64) * np.uint64(tbuf.shape[1])).astype(np.uint64)
    qlen = np.full(n, qbuf.shape[1], dtype=np.int32)
    ptrs = (qptr, qlen, tptr, tlens)
    cfg, _ = make_config(500, MODE_NW, TASK_LOC)
    cells = float((qlen.astype(np.float64) * tlens).sum())
    ee = e2e_steps(E, ptrs, n, cfg, steps, barrier, keep_last=True)
    res = ee["res"]
    rep = E.kernel_report()
    kernels_ms = {k: round(v[0], 4) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][0])}
    cs = cpu_sample({"n": n, "get": lambda i: (qbuf[i].tobytes(), tbuf[i, :tlens[i]].tobytes())}, MODE_NW, TASK_LOC, 500,
                    cpu_seconds, cores, lambda i: 10_000 * int(tlens[i]))
    checked = check_sample(res, cs["results"], "config 3")
    within = float((res["editDistance"] >= 0).mean())
    mean_ed = float(res["editDistance"][res["editDistance"] >= 0].mean())
    E.free(res)
    t = float(np.mean(ee["times"]))
    dom = next(iter(kernels_ms)) if kernels_ms else None
    dom_s = kernels_ms.get(dom, 0.0) / 1e3
    bytes_alg = float(qlen.sum()) + float(tlens.sum()) + 16.0 * n  # SURVEY.md 8d: query + target + distance/locations
    return {"workload": "configs[2]: %d pairs, 10 kbp query vs its 3 %%-mutated copy, NW, k=500, EDLIB_TASK_LOC" % n,
            "generation_s": gen_s, "e2e": {"pairs_per_s": n / t, "gcups": cells / t / 1e9, "ms_per_batch": 1000 * t,
                                           "h2d_bytes": ee["h2d"], "d2h_bytes": ee["d2h"]},
            "kernel_ms": ee["kernel_ms"], "kernels_ms": kernels_ms,
            "roofline": {"bound": "hbm", "kernel": dom, "kernel_ms": dom_s * 1e3, "bytes_algorithmic": bytes_alg,
                         "achieved": bytes_alg / dom_s / 1e9 if dom_s > 0 else None, "peak": peak, "unit": "GB/s",
                         "frac": bytes_alg / dom_s / 1e9 / peak if dom_s > 0 else None, "peak_source": peak_src,
                         "note": "algorithmic bytes = every query + every target + 16 B of results, over the device time of the "
                                 "dominant kernel; end to end the batch is bound by its %.1f GB host->device copy" % (ee["h2d"] / 1e9)},
            "cpu_baseline": {"pairs_per_s": cs["alignments_per_s"], "gcups": cs["gcups"], "cores": cores, "kind": cs["kind"],
                             "sample": "first %d pairs, %.1f s wall; every result field bit-exact vs the GPU" % (checked, cs["wall"])},
            "fraction_within_k": within, "mean_edit_distance": mean_ed}


def config4(E, target, reads, steps, cores, cpu_seconds, barrier, peak=None, peak_src=None):
    """BASELINE configs[3]: the headline batch with EDLIB_TASK_PATH, plus the extended CIGAR of every alignment."""
    n = reads.shape[0]
    ptrs = pointer_arrays(reads, target)
    cfg, _ = make_config(-1, MODE_HW, TASK_PATH)
    import torch
    times, cigar_times = [], []
    res = cg = None
    for it in range(1 + steps):
        if res is not None:
            E.free_cigars(cg)
            E.free(res)
        res = np.empty(n, dtype=RESULT_DTYPE)
        res.view(np.uint8).fill(0)
        barrier()
        t0 = time.perf_counter()
        E.align_batch(ptrs, n, cfg, res)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        cg = E.cigars(res)
        t2 = time.perf_counter()
        if it > 0:
            times.append(t2 - t0)
            cigar_times.append(t2 - t1)
    st = Stats()
    E.L.edlibB200LastStats(C.byref(st))
    rep = E.kernel_report()
    kernels_ms = {k: round(v[0], 4) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][0])}
    tb = target.tobytes()
    cs = cpu_sample({"n": n, "get": lambda i: (reads[i].tobytes(), tb)}, MODE_HW, TASK_PATH, -1, cpu_seconds, cores,
                    lambda i: READ_LEN * len(target), want_cigar=True)
    cig = [C.string_at(cg[i]).decode("ascii") if cg[i] else None for i in range(len(cs["results"]))]
    checked = check_sample(res, cs["results"], "config 4", cigars=cig)
    mean_aln = float(res["alignmentLength"].mean())
    nloc_sum = float(res["numLocations"].sum())
    aln_sum = float(res["alignmentLength"].sum())
    E.free_cigars(cg)
    E.free(res)
    t = float(np.mean(times))
    cells = float(n) * READ_LEN * len(target)
    return {"workload": "configs[3]: %d x %d bp reads, HW, EDLIB_TASK_PATH + edlibAlignmentToCigar(EXTENDED), vs the %d bp target"
                        % (n, READ_LEN, len(target)),
            "e2e": {"gcups": cells / t / 1e9, "alignments_per_s": n / t, "ms_per_batch": 1000 * t,
                    "cigar_ms": 1000 * float(np.mean(cigar_times)), "h2d_bytes": int(st.h2dBytes), "d2h_bytes": int(st.d2hBytes)},
            "kernel_ms": float(st.kernelMs), "kernels_ms": kernels_ms,
            "roofline": config4_roofline(kernels_ms, n, len(target), nloc_sum, aln_sum, float(st.kernelMs), peak, peak_src),
            "cpu_baseline": {"alignments_per_s": cs["alignments_per_s"], "gcups": cs["gcups"], "cores": cores, "kind": cs["kind"],
                             "sample": "first %d reads, %.1f s wall; every result field and the CIGAR bit-exact vs the GPU" % (checked, cs["wall"])},
            "mean_alignment_length": mean_aln}


def config4_roofline(kernels_ms, n, target_len, nloc_sum, aln_sum, kernel_ms, peak, peak_src):
    """Dominant kernel of the PATH batch against the HBM peak: SURVEY.md 8d's algorithmic bytes (query + whole target +
    distance / counts + 8 B per location + the edit script, per alignment) over its device time, beside the bytes the
    PATH phase must really move (stored matrices of the banded slices: written once, read once by the traceback)."""
    if not kernels_ms or not peak:
        return None
    dom = next(iter(kernels_ms))
    dom_s = kernels_ms[dom] / 1e3
    bytes_alg = float(n) * (READ_LEN + target_len + 8) + 8.0 * nloc_sum + aln_sum
    stored = float(n) * (READ_LEN + 10) * 5 * 8  # {Pv, Ph} per column and word of a ~160-column slice, 5 words
    return {"bound": "hbm", "kernel": dom, "kernel_ms": kernels_ms[dom], "bytes_algorithmic": bytes_alg,
            "achieved": bytes_alg / dom_s / 1e9 if dom_s > 0 else None, "peak": peak, "unit": "GB/s",
            "frac": bytes_alg / dom_s / 1e9 / peak if dom_s > 0 else None, "peak_source": peak_src,
            "stored_matrix_bytes": stored, "all_kernels_ms": kernel_ms,
            "note": "nominal accounting as in the headline (every alignment 'consumes' its whole target); the PATH phase itself "
                    "writes and re-reads ~%.1f GB of stored matrices, which bounds its lane / traceback kernels" % (stored / 1e9)}


def long_hw(E, genome, cores):
    """Long queries (> 256 bp, up to 10 kbp; 60 % .. 100 % identity) of the reference's E. coli test data, HW, EDLIB_TASK_LOC,
    over the 4.63 Mbp genome: each read as ONE edlibAlign call (latency), all of them as one edlibAlignBatch, and the
    reference build on the same reads (one core per read)."""
    with open(os.path.join(REPO, "tests", "golden", "ecoli_reads.json")) as f:
        fx = json.load(f)["reads"]
    names = sorted(n for n in fx if len(fx[n]["seq"]) > 256)
    seqs = [fx[n]["seq"].encode("ascii") for n in names]
    gb = genome.tobytes()
    lib, kind = ref_lib()
    cfg, _ = make_config(-1, MODE_HW, TASK_LOC)
    from edlib_b200._ffi import result_to_dict
    per = {}
    E.lib.align(seqs[0], gb, -1, MODE_HW, TASK_LOC)  # warm-up of the call path
    for n, q in zip(names, seqs):
        t0 = time.perf_counter()
        got = E.lib.align(q, gb, -1, MODE_HW, TASK_LOC)
        t1 = time.perf_counter()
        r = lib.align_raw(q, gb, cfg)
        t2 = time.perf_counter()
        exp = result_to_dict(r)
        lib.free(r)
        assert got == exp, "long HW read %s differs from the reference" % n
        per[n] = {"bp": len(q), "editDistance": got["editDistance"], "gpu_ms": 1000 * (t1 - t0), "cpu_1core_ms": 1000 * (t2 - t1),
                  "speedup_vs_1core": (t2 - t1) / (t1 - t0)}
    t0 = time.perf_counter()
    st, res = E.lib.align_batch(seqs, [gb] * len(seqs), -1, MODE_HW, TASK_LOC)
    tb = time.perf_counter() - t0
    assert st == 0
    cpu_total = sum(v["cpu_1core_ms"] for v in per.values())
    return {"workload": "%d reads of 257..10,000 bp (tests/golden/ecoli_reads.json: mason reads and their 60..99 %% mutated copies), "
                        "HW, EDLIB_TASK_LOC, vs the 4,630,707 bp genome" % len(seqs),
            "single_calls": per, "batch_ms": 1000 * tb, "sum_gpu_single_ms": sum(v["gpu_ms"] for v in per.values()),
            "sum_cpu_1core_ms": cpu_total, "cpu_kind": kind, "batch_speedup_vs_1core": cpu_total / (1000 * tb),
            "batch_speedup_vs_%d_cores_ideal" % cores: cpu_total / cores / (1000 * tb)}


def strong_scaling(E, genome, total_reads, steps, rank, world, dev, barrier):
    """BASELINE configs[4]: ONE batch of `total_reads` reads (seed 44) sharded over the ranks (sharding.shard_range).
    Inside every timed step: NCCL broadcast of the target from rank 0, edlibAlignBatch on the rank's shard (host
    buffers), gather of the per-read distances on rank 0."""
    import torch
    import torch.distributed as dist
    n_t = len(genome)
    lo, hi = sharding.shard_range(total_reads, rank, world)
    # every rank derives its shard of the seeded batch: read i only depends on (seed, i)
    reads = workloads.pinned_empty((hi - lo, READ_LEN), numa_node=E.numa_node)
    workloads._synth().synth_reads_range(genome.ctypes.data, n_t, reads.ctypes.data, lo, hi, READ_LEN, 0.03, 44)
    cfg, _ = make_config(-1, MODE_HW, TASK_DISTANCE)
    times = []
    mean_ed = None
    # buffers that live across the steps: the rank's copy of the target (pinned: one address, so the pointer arrays are
    # built once), the gathered distances on rank 0
    tbuf = workloads.pinned_empty((n_t,), numa_node=E.numa_node)
    if world == 1:
        tbuf[:] = genome
    ptrs = pointer_arrays(reads, tbuf)
    counts = [sharding.shard_range(total_reads, r, world)[1] - sharding.shard_range(total_reads, r, world)[0] for r in range(world)]
    all_out = workloads.pinned_empty((total_reads,), dtype=np.int32, numa_node=E.numa_node) if (rank == 0 and world > 1) else None
    for it in range(1 + steps):
        res = np.empty(hi - lo, dtype=RESULT_DTYPE)
        res.view(np.uint8).fill(0)
        barrier()
        t0 = time.perf_counter()
        if world > 1:
            sharding.broadcast_target_into(genome if rank == 0 else None, tbuf, dev)
        E.align_batch(ptrs, hi - lo, cfg, res)
        eds = np.ascontiguousarray(res["editDistance"])
        all_eds = sharding.gather_int32_known(eds, counts, dev, out=all_out) if world > 1 else eds
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        E.free(res)
        if rank == 0:
            assert len(all_eds) == total_reads
            mean_ed = float(all_eds.mean())
        if it > 0:
            times.append(dt)
    el = torch.tensor([sum(times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    t = float(el.item()) / max(steps, 1)
    cells = float(total_reads) * READ_LEN * n_t
    return {"workload": "configs[4]: %d x %d bp reads (seed 44), HW distance, one batch sharded over %d rank(s); target broadcast "
                        "(NCCL) + edlibAlignBatch from host buffers + gather of the distances inside the step" % (total_reads, READ_LEN, world),
            "scaling": "strong", "n_gpus": world, "steps": steps, "ms_per_step": 1000 * t, "gcups": cells / t / 1e9,
            "alignments_per_s": total_reads / t, "mean_edit_distance": mean_ed}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = effective_cores()
    target = workloads.ecoli_genome() if args.target == "ecoli" else workloads.random_dna(SYNTH_TARGET_LEN, 1)
    reads = workloads.reads_of(target, min(args.reads, 200_000), READ_LEN, seed=42)
    tb = target.tobytes()
    per_step_goal = max(1.0, min(6.0, 60.0 / max(1, args.warmup + args.steps)))  # the whole run stays near a minute
    times, samples, kind = [], [], "reference"
    for step in range(args.warmup + args.steps):
        cs = cpu_sample({"n": len(reads), "get": lambda i: (reads[i].tobytes(), tb)}, MODE_HW, TASK_DISTANCE, -1, per_step_goal,
                        cores, lambda i: READ_LEN * len(target))
        kind = cs["kind"]
        if step >= args.warmup:
            times.append(cs["wall"])
            samples.append(cs["sample"])
    cells = sum(samples) * READ_LEN * len(target)
    total = sum(times)
    value = cells / total / 1e9
    line = {
        "impl": "reference", "metric": "GCUPS", "value": value, "unit": "GCUPS (nominal cells/s / 1e9)",
        "alignments_per_s": sum(samples) / total, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "configs[1]: %d bp reads HW distance k=-1 vs one %d bp target (%s); each step = bounded sample of "
                               "%d reads of the same batch on %d host cores" % (READ_LEN, len(target), args.target, samples[-1], cores)},
        "cpu_baseline": {"value": value, "unit": "GCUPS", "cores": cores, "gcups_per_core": value / cores, "kind": kind,
                         "sample": "%d reads per step x %d steps" % (samples[-1], args.steps)},
        "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per GPU (default: the named config)")
    ap.add_argument("--target", default="ecoli", choices=["ecoli", "synthetic"],
                    help="ecoli: the 4,630,707 bp E. coli DH1 genome (BASELINE configs[1]); synthetic: uniform-random 5,000,000 bp")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep-sample", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sub-records (other configs, sensitivity, strong scaling)")
    ap.add_argument("--extras", default="strong,target_handle,other_target,sensitivity,long_hw,config4,config3,sweep_kernel",
                    help="comma-separated sub-records to run (default: all)")
    ap.add_argument("--config3-pairs", type=int, default=100_000)
    ap.add_argument("--strong-reads", type=int, default=10_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step of the headline workload to DIR/<name>.npy (dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the one JSON line: whatever NCCL_DEBUG level is set goes to a file
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/nccl_debug_%h_%p.log")
        dist.init_process_group("nccl", device_id=dev)
    E = Engine(local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def flush_l2():
        flush_buf.zero_()
        torch.cuda.synchronize()

    # ---- workload: shared target from rank 0 (one NCCL broadcast), own shard of reads per rank ----
    n_reads = args.reads
    if rank == 0:
        target = workloads.ecoli_genome() if args.target == "ecoli" else workloads.random_dna(SYNTH_TARGET_LEN, 1)
    else:
        target = None
    t_len = 4_630_707 if args.target == "ecoli" else SYNTH_TARGET_LEN
    if world > 1:
        target = sharding.broadcast_target(target, t_len, dev)
    E_numa = E.numa_node
    pinned_target = workloads.pinned_empty((t_len,), numa_node=E_numa)  # the genome too sits in pinned host memory
    pinned_target[:] = target
    target = pinned_target
    reads = workloads.reads_of(target, n_reads, READ_LEN, seed=42 + rank, pinned=True, numa_node=E.numa_node)
    cells_rank = float(n_reads) * READ_LEN * t_len
    cores = effective_cores()

    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    sampler = ClockSampler(range(local_world)) if rank == 0 else None
    if sampler:
        sampler.start()
    rs, ee, eds, nloc, cpu = run_reads_workload(E, target, reads, args.steps, args.warmup, args.e2e_steps, flush_l2, barrier,
                                                want_cpu=(cores if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None),
                                                cpu_seconds=args.cpu_seconds,
                                                dump=(args.dump_outputs, "rank%d_" % rank if world > 1 else "") if args.dump_outputs else None)
    all_clocks = sampler.stop() if sampler else {}
    clocks = all_clocks.get(local_rank)
    elapsed = torch.tensor([sum(rs["step_s"])], dtype=torch.float64, device=dev)
    e2e_t = torch.tensor([sum(ee["times"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(elapsed, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        all_eds = sharding.gather_int32(eds, dev)  # (the gather of results on rank 0; timed in `strong`)
        if rank == 0:
            assert len(all_eds) == world * n_reads
    per_rank = None
    if world > 1:  # what every rank saw (the slowest one sets the value): step time, device time of its kernels, e2e step
        mine = torch.tensor([1000.0 * sum(rs["step_s"]) / max(args.steps, 1), rs["kernel_ms"],
                             1000.0 * sum(ee["times"]) / max(args.e2e_steps, 1)], dtype=torch.float64, device=dev)
        allr = [torch.zeros(3, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": r, "ms_per_step": float(t[0]), "kernel_ms_per_step": float(t[1]), "e2e_ms_per_step": float(t[2]),
                     "clocks": all_clocks.get(r)} for r, t in enumerate(allr)]
    elapsed = float(elapsed.item())
    e2e_value = (world * cells_rank * args.e2e_steps / float(e2e_t.item()) / 1e9) if args.e2e_steps > 0 else None

    line = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        value = world * cells_rank * args.steps / elapsed / 1e9
        line = {
            "metric": "GCUPS", "value": value, "unit": "GCUPS (nominal cells/s / 1e9)",
            "alignments_per_s": world * n_reads * args.steps / elapsed,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * elapsed / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "configs[1]: %d x %d bp reads (3%% sub/ins/del, seeded), HW, EDLIB_TASK_DISTANCE, k=-1, vs one %d bp "
                                   "target (%s), per GPU" % (n_reads, READ_LEN, t_len,
                                                             "E. coli DH1 genome of the reference's test data" if args.target == "ecoli"
                                                             else "uniform-random DNA, seed 1"),
                       "inputs": "the read array lives in pinned host memory (torch pin_memory) on the GPU's NUMA node (node %d); "
                                 "end-to-end calls upload it from there (no staging copy); results are malloc'd arrays per read "
                                 "as in the reference" % E.numa_node,
                       "host_allocator": "glibc told to keep freed memory (edlibB200TuneHostAllocator: mallopt M_TRIM_THRESHOLD / "
                                         "M_TOP_PAD): %s" % E.allocator_tuned,
                       "l2": "256 MiB write between steps (reads 150 MB > L2; the target is meant to stay L2-resident)",
                       "parallelism": "reads sharded over %d rank(s); target broadcast once" % world,
                       "index": "the seed index of the target is rebuilt inside every timed step (no target handle)"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": ee["h2d"], "d2h_bytes_per_step": ee["d2h"],
                    "ms_per_step": 1000.0 * float(e2e_t.item()) / max(args.e2e_steps, 1), "kernel_ms_last_step": ee["kernel_ms"]},
            "gpu_launches": int(rs["launches"]),
            "roofline": reads_roofline(rs, n_reads, t_len, float(nloc.sum()), sm_mhz, peak, peak_src),
            "cpu_baseline": cpu,
            "mean_edit_distance": float(eds.mean()), "mean_num_locations": float(nloc.mean()),
            "filter": rs["filter"], "kernel_ms_per_step": rs["kernel_ms"],
            "kernel_share_of_step": rs["kernel_ms"] / (1000.0 * elapsed / args.steps),
            "per_rank": per_rank,
        }
    # ---- strong scaling (configs[4]) on every N; the other sub-records on one GPU only ----
    wanted = set() if args.no_extras else set(x for x in args.extras.split(",") if x)
    if "strong" in wanted:
        try:
            genome = target if args.target == "ecoli" else (workloads.ecoli_genome() if rank == 0 else None)
            if world > 1 and args.target != "ecoli":
                genome = sharding.broadcast_target(genome, 4_630_707, dev)
            s = strong_scaling(E, genome, args.strong_reads, 3, rank, world, dev, barrier)
            if line is not None:
                line["strong"] = s
        except Exception as e:  # a sub-record never takes the headline down
            if line is not None:
                line["strong"] = {"error": repr(e)[:300]}
    if rank == 0 and world == 1 and wanted:
        peak, peak_src = measured_peaks()
        extras = {}

        def guarded(name, fn):
            if name not in wanted:
                return
            t0 = time.time()
            try:
                extras[name] = fn()
            except AssertionError:
                raise  # a parity failure is never swallowed
            except Exception as e:
                extras[name] = {"error": repr(e)[:300]}
            if isinstance(extras[name], dict):
                extras[name]["wall_s"] = round(time.time() - t0, 1)

        def synthetic():
            other = workloads.random_dna(SYNTH_TARGET_LEN, 1) if args.target == "ecoli" else workloads.ecoli_genome()
            rd = workloads.reads_of(other, n_reads, READ_LEN, seed=42, pinned=True, numa_node=E.numa_node)
            r2, e2, ed2, nl2, _ = run_reads_workload(E, other, rd, 5, 2, 3, flush_l2, barrier)
            c = float(n_reads) * READ_LEN * len(other)
            return {"target": "uniform-random 5,000,000 bp (seed 1)" if args.target == "ecoli" else "E. coli DH1 (4,630,707 bp)",
                    "value": c * 5 / sum(r2["step_s"]) / 1e9, "ms_per_step": 1000 * float(np.mean(r2["step_s"])),
                    "e2e": {"value": c * 3 / sum(e2["times"]) / 1e9, "ms_per_step": 1000 * float(np.mean(e2["times"]))},
                    "kernel_ms_per_step": r2["kernel_ms"], "kernels_ms": r2["kernels_ms"], "filter": r2["filter"],
                    "mean_edit_distance": float(ed2.mean())}

        def target_handle():
            # the headline batch again, end to end, against a target kept resident (include/edlib_b200.h:
            # edlibB200TargetPrepare): upload, encoding and seed index of the target are paid once, outside the steps
            t0 = time.perf_counter()
            h = E.L.edlibB200TargetPrepare(target.ctypes.data, len(target))
            assert h, E.L.edlibB200LastError()
            prep = time.perf_counter() - t0
            cfg, _ = make_config(-1, MODE_HW, TASK_DISTANCE)
            ee2 = e2e_steps(E, pointer_arrays(reads, target), n_reads, cfg, 5, barrier, expect_ed=eds)
            E.L.edlibB200TargetFree(h)
            t = float(np.mean(ee2["times"]))
            return {"note": "edlibAlignBatch against a target registered with edlibB200TargetPrepare (index NOT rebuilt per step; "
                            "distances identical to the headline's)", "prepare_ms": 1000 * prep,
                    "e2e": {"value": cells_rank / t / 1e9, "ms_per_step": 1000 * t, "h2d_bytes_per_step": ee2["h2d"],
                            "d2h_bytes_per_step": ee2["d2h"]}}

        guarded("target_handle", target_handle)
        guarded("other_target", synthetic)
        guarded("sensitivity", lambda: sensitivity(E, target, reads, flush_l2, barrier))
        guarded("long_hw", lambda: long_hw(E, target if args.target == "ecoli" else workloads.ecoli_genome(), cores))
        guarded("config4", lambda: config4(E, target, reads, 2, cores, 10.0, barrier, peak, peak_src))
        del reads
        genome = target if args.target == "ecoli" else workloads.ecoli_genome()
        guarded("config3", lambda: config3(E, genome, args.config3_pairs, 2, cores, 10.0, peak, peak_src, barrier))
        if not args.no_sweep_sample:
            guarded("sweep_kernel", sweep_kernel_sample)
        line.update(extras)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
