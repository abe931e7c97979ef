#!/usr/bin/env python
"""bench.py — headline benchmark of the arrow-go compute hot path on B200.

Workload (BASELINE.json configs[1]): compute.Add(float64, float64) on a 100M-row CHUNKED array
per GPU (left: 100 chunks of 1M rows; right: chunks of 999,983 rows so the executor's span
iteration sees misaligned chunk boundaries, arrow/compute/executor.go:757-863), one contiguous
preallocated output (executor.go:598-623).  A "step" is one Add over the whole column.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

ONE JSON line on rank 0 (contract in the task statement):
  value     rows/s, whole job (all ranks), kernels timed with CUDA events on device-resident
            buffers (1.6 GB in + 0.8 GB out per step: far larger than the 126 MB L2, so no flush)
  e2e       same metric through the HOST-pointer C ABI (ag_arith_binary on pinned host buffers):
            H2D of both inputs and D2H of the result inside the timed region
  roofline  achieved HBM GB/s of the Add kernel = 24 B/row x rows / CUDA-event time, against
            MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference's own AVX2 loop (oracle/_ref, assembled from the reference's
            checked-in assembly) on a bounded sample of the same workload, 1 thread — what a
            reference CallFunction uses (arrow/compute/exec.go:164-170) — plus an all-cores
            row-sharded figure for context
  others    kernel-only numbers for Sum / Greater / Filter / fused / Take at 100M rows, Add on sliced (element-aligned)
            operands, the reference-order Sum mode, the global Sum (mailbox and NCCL forms), BASELINE configs 4 and 5
            at their full 1B rows split over the ranks (values asserted), PCIe peaks and the config-3 resident pipeline
`--impl reference` times the reference's CPU path alone (same metric, same config): the full 100M-row chunked Add per
step, one pinned core, span loop and clock in C (oracle/bench_cpu.c).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS = 100_000_000
L_CHUNK = 1_000_000
R_CHUNK = 999_983
METRIC = "rows/sec, compute.Add(float64,float64) on a 100M-row chunked array per GPU"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the Add kernel from the committed
    `ncu --set full` capture (profiles/r2/ncu_full_bench_kernels.csv), or None."""
    import csv
    path = os.path.join(ROOT, "profiles", "r2", "ncu_full_bench_kernels.csv")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r1", "ncu_full_binary_spans_kernel.csv")
    try:
        rows = list(csv.reader(open(path)))
        h = rows[0]
        ri = [i for i, c in enumerate(h) if c.startswith("dram__bytes_read.sum")][0]
        wi = [i for i, c in enumerate(h) if c.startswith("dram__bytes_write.sum")][0]
        scale = lambda c: {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[c[c.index("[") + 1:c.index("]")]]
        vals = [float(r[ri]) * scale(h[ri]) + float(r[wi]) * scale(h[wi]) for r in rows[1:]]
        return sum(vals) / len(vals)
    except Exception:
        return None


def spans_for(n, lc, rc):
    """iterateExecSpans (executor.go:757-863): span = min(remaining of each arg's current chunk)."""
    out, pos = [], 0
    while pos < n:
        l_rem = lc - pos % lc
        r_rem = rc - pos % rc
        ln = min(l_rem, r_rem, n - pos)
        out.append((pos, ln))
        pos += ln
    return out


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md).  NVML is
    polled from a thread every few ms (nvidia-smi's 100 ms loop is too coarse for a 10-40 ms
    timed region); nvidia-smi is the fallback when pynvml is unavailable."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device):
        self.device = device
        self.samples, self.max_mhz, self.reasons = [], None, set()
        self._stop = threading.Event()
        self._t = None
        self._nvml = None

    def _loop(self):
        nv, h = self._nvml, self._h
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self._nvml = nv
            self._h = nv.nvmlDeviceGetHandleByIndex(self.device)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        except Exception:
            self._nvml = None

    def stop(self):
        if self._nvml is None:
            return self._smi_once()
        self._stop.set()
        self._t.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_min_mhz": float(min(self.samples)), "sm_max_mhz": float(self.max_mhz),
                "reasons": sorted(self.reasons), "samples": len(self.samples), "source": "nvml, 2 ms poll during the timed regions"}

    def _smi_once(self):
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.device}", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 1, "source": "nvidia-smi (idle snapshot)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}


# ------------------------------------------------------------------ reference / CPU arm -----
def bench_config(rows, world):
    """The `config` object, identical for both arms."""
    return {"workload": "compute.Add(float64,float64) on a 100M-row chunked array per GPU (BASELINE.json configs[1])",
            "rows_per_gpu": rows, "chunks": f"left {L_CHUNK}-row chunks, right {R_CHUNK}-row chunks -> {len(spans_for(rows, L_CHUNK, R_CHUNK))} spans, one contiguous output",
            "l2": "inputs (1.6 GB) + output (0.8 GB) per step exceed the 126 MB L2 (and every CPU cache); no flush needed",
            "parallelism": f"row-range x{world}"}


class CpuAdd:
    """The reference's own inner loop for this config — _arithmetic_binary_avx2(FLOAT64, OpAddChecked, l, r, out, len)
    (base_arithmetic_avx2_amd64.go:35-39) called once per span like executeSpans does (executor.go:598-623) — timed by
    the C harness oracle/bench_cpu.c: span loop and clock_gettime in C, the thread pinned to one core."""

    def __init__(self, rows):
        from oracle import oracle
        self.rows = rows
        self.h = oracle.bench()
        ref = oracle.ref()
        self.isa = oracle.host_isa()
        if ref is not None:
            self.fn = C.cast(getattr(ref, f"arithmetic_binary_{self.isa}"), C.c_void_p)
            self.kind = "reference"
        else:
            self.fn = C.cast(oracle.cpu().ref_arith_binary_native_abi, C.c_void_p)
            self.kind = "port"
        rng = np.random.default_rng(0x94378165)   # dataset E: integers stored as double
        self.a = rng.integers(-(1 << 20), 1 << 20, rows).astype(np.float64)
        self.b = rng.integers(-(1 << 20), 1 << 20, rows).astype(np.float64)
        self.out = np.zeros(rows)
        try:
            self.cores = sorted(os.sched_getaffinity(0))
        except AttributeError:
            self.cores = list(range(os.cpu_count() or 1))

    def _run(self, lo, hi, warmup, steps, core):
        times = (C.c_double * steps)()
        if core is not None:
            self.h.bench_pin_to_core(core)
        self.h.bench_add_f64_chunked(self.fn, 12, 21, self.a.ctypes.data, self.b.ctypes.data, self.out.ctypes.data, lo, hi,
                                     L_CHUNK, R_CHUNK, warmup, steps, times)
        return list(times)

    def one_core(self, warmup, steps):
        """rows/s over exactly `steps` timed full-size steps on one pinned core (what a reference CallFunction uses,
        arrow/compute/exec.go:164-170)."""
        saved = os.sched_getaffinity(0)
        try:
            t = self._run(0, self.rows, warmup, steps, self.cores[len(self.cores) // 2])
        finally:
            os.sched_setaffinity(0, saved)
        assert np.array_equal(self.out[:1000], self.a[:1000] + self.b[:1000]) and np.array_equal(self.out[-1000:], self.a[-1000:] + self.b[-1000:])
        return self.rows * steps / sum(t), self.rows / min(t), sum(t) / steps

    def all_cores(self, warmup, steps):
        """Context only (NOT a reference feature): the same loop row-range sharded over every host core, one pinned
        thread per core, wall clock around the whole pool."""
        T = len(self.cores)
        cuts = np.linspace(0, self.rows, T + 1).astype(np.int64)
        with ThreadPoolExecutor(T) as pool:
            list(pool.map(lambda i: self._run(int(cuts[i]), int(cuts[i + 1]), 1, 1, self.cores[i]), range(T)))   # page faults, pin
            t0 = time.perf_counter()
            list(pool.map(lambda i: self._run(int(cuts[i]), int(cuts[i + 1]), 0, steps, self.cores[i]), range(T)))
            dt = time.perf_counter() - t0
        return self.rows * steps / dt, T


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = int(os.environ.get("AG_BENCH_REF_ROWS", str(args.rows)))   # the CPU tests shrink it
    W, K = max(args.warmup, 1), max(args.steps, 1)
    t0 = time.perf_counter()
    cpu = CpuAdd(rows)
    one, one_best, s_per_step = cpu.one_core(min(W, 3), K)
    allc, T = cpu.all_cores(1, max(2, min(K, 5)))
    wall = time.perf_counter() - t0
    line = {
        "impl": "reference", "metric": METRIC, "value": one, "unit": "rows/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(rows, args.gpus),
        "cpu_baseline": {"value": one, "unit": "rows/s", "cores": 1, "kind": cpu.kind, "isa": cpu.isa, "best_step": one_best,
                         "sample": f"the full workload: {rows} rows x {K} steps, span loop + clock_gettime in C (oracle/bench_cpu.c), thread pinned to core "
                                   f"{cpu.cores[len(cpu.cores) // 2]}; the reference executes a CallFunction's spans on one goroutine (exec.go:164-170)",
                         "all_cores": {"value": allc, "unit": "rows/s", "cores": T, "note": "row-range sharded over every host core, one pinned thread each; NOT a reference feature, context only"}},
        "e2e": {"value": one, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall, "timing": "clock_gettime(CLOCK_MONOTONIC) per step inside the C harness, host resident",
    }
    _emit(line)


# ------------------------------------------------------------------ helpers of our arm -----
def _mix64_np(z):
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def full_size_configs(N, comm, dist, rank, world, peak, timed, DeviceBuffer, total_rows):
    """BASELINE configs[3] and [4]: Take(int64 values, int32 indices) with the 1B-row (8 GB) values table replicated on
    every GPU and 1B random indices sharded by row range; Int64 Sum over 1B rows sharded by row range with the global
    fold.  The results are ASSERTED: the Sum against the oracle's generator twin + wrapping sum of every rank's shard,
    the Take element by element on sampled windows (values[i] = mix64(i)), by cross-checking the windowed path's whole
    output against the direct path's through the order-sensitive device checksum, and through a planted bad index."""
    from oracle import oracle
    cpu = oracle.cpu()
    out = {}
    a, b = C.c_int64(), C.c_int64()
    N.call("ag_shard_range", total_rows, rank, world, C.byref(a), C.byref(b))
    lo, n = a.value, b.value - a.value
    scal = DeviceBuffer(64)
    # ---- C5: Int64 Sum, column = mix64(seed + global row) (full range, wraps)
    col = DeviceBuffer(max(n, 1) * 8)
    N.call("ag_generate_dev", 0, 0x94378165 + lo, 0, 0, col.ptr, n, None)
    ms_local = timed(lambda: N.call("ag_sum_i64_dev", col.ptr, n, scal.ptr, None), 3, 10)
    ms = timed(lambda: N.call("ag_sum_i64_global_dev", comm, col.ptr, n, scal.ptr, None), 3, 10)
    N.call("ag_stream_sync", None)
    got = int(scal.to_numpy(np.int64, 1)[0])
    want, chunk = 0, 1 << 26
    tmp = np.empty(chunk, dtype=np.uint64)
    for off in range(0, n, chunk):
        m = min(chunk, n - off)
        cpu.ref_generate(0, 0x94378165 + lo + off, 0, 0, tmp.ctypes.data, m)
        want = (want + cpu.ref_sum_i64(tmp.ctypes.data, m)) % (1 << 64)
    if dist is not None:
        import torch
        t = torch.tensor([want - (1 << 64) if want >= 1 << 63 else want], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)   # wrapping int64 sum of the per-rank expected values (verification plumbing only)
        want = int(t.item()) % (1 << 64)
    assert got % (1 << 64) == want, f"config 5: global Sum {got} != expected {want}"
    out["config5_sum_i64_1b_rows"] = {"total_rows": total_rows, "rows_per_gpu": n, "ranks": world, "ms": ms, "ms_local_sum_only": ms_local,
                                      "rows_per_s": total_rows / ms * 1e3, "gbs_per_gpu": 8.0 * n / ms / 1e6, "frac": 8.0 * n / ms / 1e6 / peak,
                                      "verified": "global value == wrapping sum of the oracle's generator twin over all 1B rows",
                                      "note": "row-range shards (ag_shard_range), Sum + cross-GPU fold in one kernel (ag_sum_i64_global_dev)"}
    col.free()
    # ---- C4: Take
    table_rows = total_rows
    table = DeviceBuffer(table_rows * 8); idx = DeviceBuffer(max(n, 1) * 4); o = DeviceBuffer(max(n, 1) * 8); bad = DeviceBuffer(64); ck = DeviceBuffer(64)
    N.call("ag_generate_dev", 0, 0, 0, 0, table.ptr, table_rows, None)                                   # values[i] = mix64(i)
    N.call("ag_generate_dev", 2, 0x0FF1CE + lo, 0, min(table_rows, 1 << 31) - 1, idx.ptr, n, None)      # uniform in [0, table_rows)
    N.call("ag_error_word_reset_dev", bad.ptr, None)
    take = lambda: N.call("ag_take_primitive_dev", 64, table.ptr, None, 0, table_rows, 32, 1, idx.ptr, None, 0, n, 1, o.ptr, None, bad.ptr, None)
    ms = timed(take, 2, 5)
    N.call("ag_checksum64_dev", o.ptr, n, ck.ptr, None)
    N.call("ag_stream_sync", None)
    ck_windowed = int(ck.to_numpy(np.uint64, 1)[0])
    win, checked = min(4_000_000, n), 0
    for start in (0, n // 3, n - win):
        ii = idx.to_numpy(np.int32, win, start * 4)
        oo = o.to_numpy(np.uint64, win, start * 8)
        assert np.array_equal(oo, _mix64_np(ii.astype(np.uint64))), f"config 4: take mismatch in the window at row {lo + start}"
        checked += win
    assert int(bad.to_numpy(np.int64, 1)[0]) == (1 << 63) - 1
    N.call("ag_take_set_policy", 1, 0, 0, 0)       # the one-pass gather on the same inputs: whole-output cross-check
    ms_direct = timed(take, 1, 2)
    N.call("ag_take_set_policy", 0, 0, 0, 0)
    N.call("ag_checksum64_dev", o.ptr, n, ck.ptr, None)
    N.call("ag_stream_sync", None)
    assert int(ck.to_numpy(np.uint64, 1)[0]) == ck_windowed, "config 4: windowed and direct paths disagree"
    pos = n // 2 + 17
    N.call("ag_upload", idx.ptr + pos * 4, np.array([-1], dtype=np.int32).ctypes.data, 4, None)
    take()
    N.call("ag_stream_sync", None)
    assert int(bad.to_numpy(np.int64, 1)[0]) == pos, "config 4: planted out-of-range index not reported at its row"
    out["config4_take_1b_rows"] = {"total_rows": total_rows, "rows_per_gpu": n, "table_rows": table_rows, "ranks": world, "ms": ms, "ms_direct_path": ms_direct,
                                   "rows_per_s": total_rows / ms * 1e3, "gbs_per_gpu": 20.0 * n / ms / 1e6, "frac": 20.0 * n / ms / 1e6 / peak,
                                   "verified": f"{checked} rows per rank element by element (values[i] = mix64(i)); whole output: checksum(windowed) == checksum(direct); planted bad index found at its row",
                                   "note": "8 GB values table replicated per GPU, indices row-range sharded, no collective (SURVEY 8e)"}
    for buf in (table, idx, o, bad, ck, scal):
        buf.free()
    return out


def link_peaks(N, h_src, h_dst, d_a, d_b, nbytes, Event, barrier, max_over_ranks):
    """Pinned-host <-> HBM copy rates of THIS box, measured beside the e2e number: H2D alone, D2H alone, both at once
    on two streams (what the host-pointer pipeline does).  Every rank copies at the same time, so at N > 1 these are
    the per-GPU rates under contention for the host's root complexes."""
    from arrow_go_b200.device import Stream
    s1, s2 = Stream(), Stream()

    def run(h2d, d2h, reps=3):
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if h2d:
                N.call("ag_upload", d_a.ptr, h_src.ptr, nbytes, s1.handle)
            if d2h:
                N.call("ag_download", h_dst.ptr, d_b.ptr, nbytes, s2.handle)
        s1.sync(); s2.sync()
        dt = max_over_ranks(time.perf_counter() - t0)
        return (int(h2d) + int(d2h)) * nbytes * reps / dt / 1e9
    run(True, True, 1)
    out = {"h2d_gbs": run(True, False), "d2h_gbs": run(False, True), "bidirectional_gbs": run(True, True), "bytes_per_copy": nbytes}
    s1.close(); s2.close()
    return out


def c3_pipeline(N, h_vals, h_out, d_vals, d_out, rows, rank, Event, barrier, max_over_ranks):
    """BASELINE config 3 end to end the way the design intends it: the int64 column is uploaded ONCE (pinned host ->
    HBM), Greater(v, 89) + Filter run fused on the resident column, only the ~10 % selected rows (80 MB) come back.
    Reported: the one-off upload, and the steady-state step (kernel + D2H of the result) on the resident column."""
    scal = None
    from arrow_go_b200.device import DeviceBuffer
    scal = DeviceBuffer(64)
    N.call("ag_generate_dev", 1, 0x0FF1CE + rank * rows, 0, 99, d_vals.ptr, rows, None)
    N.call("ag_download", h_vals.ptr, d_vals.ptr, rows * 8, None)
    N.call("ag_stream_sync", None)
    sc = np.array([89], dtype=np.int64)
    barrier()
    t0 = time.perf_counter()
    N.call("ag_upload", d_vals.ptr, h_vals.ptr, rows * 8, None)
    N.call("ag_stream_sync", None)
    t_up = max_over_ranks(time.perf_counter() - t0)

    def step():
        N.call("ag_filter_compare_scalar_dev", N.INT64, N.CMP_GT, d_vals.ptr, sc.ctypes.data, rows, d_out.ptr, rows, scal.ptr, None)
        N.call("ag_stream_sync", None)
        cnt = int(scal.to_numpy(np.int64, 1)[0])
        N.call("ag_download", h_out.ptr, d_out.ptr, cnt * 8, None)
        N.call("ag_stream_sync", None)
        return cnt
    cnt = step()
    barrier()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        cnt = step()
    t_step = max_over_ranks(time.perf_counter() - t0) / reps
    hv = np.frombuffer((C.c_char * (rows * 8)).from_address(h_vals.ptr), dtype=np.int64, count=1 << 20)
    ho = np.frombuffer((C.c_char * (rows * 8)).from_address(h_out.ptr), dtype=np.int64, count=int((hv > 89).sum()))
    assert np.array_equal(ho, hv[hv > 89]), "config 3 pipeline: filtered rows differ"
    scal.free()
    return {"rows": rows, "selected_rows": cnt, "upload_once_ms": t_up * 1e3, "upload_gbs": rows * 8 / t_up / 1e9,
            "resident_step_ms": t_step * 1e3, "resident_rows_per_s": rows / t_step, "d2h_bytes_per_step": cnt * 8,
            "first_call_ms": (t_up + t_step) * 1e3, "first_call_rows_per_s": rows / (t_up + t_step),
            "note": "Greater(int64, 89) + Filter fused (ag_filter_compare_scalar_dev) on the resident column; wall clock incl. the count readback and the D2H of the selected rows"}


DUMP_NAME = "add_f64_chunked_output"
DUMP_ROWS = 1 << 20   # 8 MB of float64
DUMP_SEED = 0xD0770


def dump_outputs(out_dir, out):
    """Rows of the Add output sampled without replacement by a fixed seed, so two builds given the same arguments
    write comparable files."""
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(out.size, min(DUMP_ROWS, out.size), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, DUMP_NAME + ".npy"), out[rows])


# ------------------------------------------------------------------ our arm ---------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=ROWS)
    ap.add_argument("--no-others", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-full-configs", action="store_true", help="skip BASELINE configs 4/5 at 1B rows")
    ap.add_argument("--full-rows", type=int, default=1_000_000_000, help="total rows of configs 4/5 (split over the ranks)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write rank 0's Add output of the last "
                    f"step as DIR/{DUMP_NAME}.npy (float64, a fixed seeded sample of {DUMP_ROWS} rows, ascending)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        # keep stdout to the ONE JSON line: NCCL writes its version banner / debug lines to stdout by
        # default; send them to stderr instead (the level the caller asked for is left alone)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from arrow_go_b200 import _native as N
    from arrow_go_b200.device import DeviceBuffer, Event, PinnedArray

    N.call("ag_init", local_rank)
    from arrow_go_b200 import sharding
    comm = sharding.create_comm(dist, device="cuda") if dist is not None else sharding.create_comm(None)
    have_nccl = False
    if dist is not None:
        try:
            sharding.attach_nccl(comm, dist, device="cuda")
            have_nccl = True
        except Exception as e:  # no libnccl.so.2 the product can dlopen: the mailbox form still runs
            print(f"rank {rank}: NCCL attach failed: {e}", file=sys.stderr)
    rows = args.rows
    W, K = max(args.warmup, 3), args.steps
    peak, peak_kind = peaks()

    def barrier():
        N.call("ag_stream_sync", None)
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident record batch (seeds SURVEY §8d; each rank its own row range) ----
    dl, dr, dout = DeviceBuffer(rows * 8), DeviceBuffer(rows * 8), DeviceBuffer(rows * 8)
    N.call("ag_generate_dev", 3, 0x94378165 + rank * rows, -(1 << 20), 1 << 20, dl.ptr, rows, None)
    N.call("ag_generate_dev", 3, 0x94378166 + rank * rows, -(1 << 20), 1 << 20, dr.ptr, rows, None)
    spans = spans_for(rows, L_CHUNK, R_CHUNK)
    launches0 = N.raw().ag_kernel_launch_count()

    # the whole chunked call is ONE launch: the span table goes to the batched entry point a
    # compute.Function that sees ChunkedDatums binds (include/arrowgpu.h: ag_arith_binary_spans_dev)
    table = N.span_table([(dl.ptr + 8 * pos, dr.ptr + 8 * pos, dout.ptr + 8 * pos, ln) for pos, ln in spans])

    def add_step():
        N.call("ag_arith_binary_spans_dev", N.FLOAT64, N.OP_ADD_CHECKED, N.SHAPE_AA, table, len(spans), None)

    def add_step_per_span():  # what a per-span exec.ArrayKernelExec binding would do (context only)
        for pos, ln in spans:
            N.call("ag_arith_binary_dev", N.FLOAT64, N.OP_ADD_CHECKED, N.SHAPE_AA, dl.ptr + 8 * pos, dr.ptr + 8 * pos, dout.ptr + 8 * pos, ln, None)

    def timed(fn, warm, steps):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = Event(), Event()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        e1.sync()
        barrier()
        return max_over_ranks(e0.elapsed_ms(e1)) / steps

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = N.raw().ag_kernel_launch_count()
    ms_chunked = timed(add_step, W, K)
    launches_timed = (N.raw().ag_kernel_launch_count() - l0) * K // (W + K)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dout.to_numpy(np.float64, rows))
    ms_per_span = timed(add_step_per_span, 3, max(3, K // 4))
    ms_contig = timed(lambda: N.call("ag_arith_binary_dev", N.FLOAT64, N.OP_ADD_CHECKED, N.SHAPE_AA, dl.ptr, dr.ptr, dout.ptr, rows, None), W, K)

    # parity spot check inside the bench (oracle = checker only): first 64K rows of the last step
    if rank == 0:
        from oracle import oracle
        a = dl.to_numpy(np.float64, 1 << 16); b = dr.to_numpy(np.float64, 1 << 16)
        want = np.empty(1 << 16)
        oracle.cpu().ref_arith_binary(12, 21, 0, a.ctypes.data, b.ctypes.data, want.ctypes.data, 1 << 16)
        assert dout.to_numpy(np.float64, 1 << 16).tobytes() == want.tobytes(), "bench output differs from the oracle"

    value = world * rows / (ms_chunked * 1e-3)
    algo_bytes = 24.0 * rows
    achieved = algo_bytes / (ms_chunked * 1e-3) / 1e9

    # ---- other kernels of the path (kernel-only, device resident) ----
    others = {}
    if not args.no_others:
        scal = DeviceBuffer(64)
        ms = timed(lambda: N.call("ag_sum_f64_dev", dl.ptr, rows, scal.ptr, None), W, K)
        others["sum_f64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 8.0 * rows / ms / 1e6, "frac": 8.0 * rows / ms / 1e6 / peak, "ms": ms}
        ms = timed(lambda: N.call("ag_sum_i64_dev", dl.ptr, rows, scal.ptr, None), W, K)
        others["sum_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 8.0 * rows / ms / 1e6, "frac": 8.0 * rows / ms / 1e6 / peak, "ms": ms}
        # reference-order mode (bit-exact AVX2 association, one warp, latency-bound by design) next to the default
        ms = timed(lambda: N.call("ag_sum_f64_reforder_dev", dl.ptr, 8192, scal.ptr, None), W, K)
        ms_def = timed(lambda: N.call("ag_sum_f64_dev", dl.ptr, 8192, scal.ptr, None), W, K)
        others["sum_f64_8192_rows"] = {"mode_default_ms": ms_def, "mode_reference_order_ms": ms, "note": "BASELINE configs[0] size; launch-bound (the reference's cache-resident loop: ~0.7-2 us)"}
        ms = timed(lambda: N.call("ag_sum_f64_reforder_dev", dl.ptr, rows, scal.ptr, None), 1, 2)
        others["sum_f64_reference_order_mode"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 8.0 * rows / ms / 1e6, "frac": 8.0 * rows / ms / 1e6 / peak, "ms": ms,
                                                  "note": "ag_sum_f64_reforder: 32 serial chains = the AVX2 order bit for bit; n/32 dependent adds, a parity tool not a fast path"}
        others["sum_f64"]["mode"] = "default: compensated (TwoSum) fixed tree, <= 1 ULP from the exactly rounded sum"
        # global Sum over the ranks: the fold is fused into the Sum kernel (HBM mailboxes over NVLink); NCCL form beside it
        ms = timed(lambda: N.call("ag_sum_i64_global_dev", comm, dl.ptr, rows, scal.ptr, None), W, K)
        others["sum_i64_global_mailbox"] = {"rows_per_s": world * rows / ms * 1e3, "ms": ms, "ranks": world,
                                            "note": "per-GPU Sum + cross-GPU fold in ONE kernel (peer stores into HBM mailboxes, rank-order fold); CUDA events, max over ranks, no host sync"}
        ms = timed(lambda: N.call("ag_sum_f64_global_dev", comm, dl.ptr, rows, scal.ptr, None), W, K)
        others["sum_f64_global_mailbox"] = {"rows_per_s": world * rows / ms * 1e3, "ms": ms, "ranks": world}
        if have_nccl:
            ms = timed(lambda: N.call("ag_sum_i64_global_nccl_dev", comm, dl.ptr, rows, scal.ptr, None), W, K)
            others["sum_i64_global_nccl"] = {"rows_per_s": world * rows / ms * 1e3, "ms": ms, "ranks": world,
                                             "note": "per-GPU Sum + ncclAllReduce(8 bytes) issued by libarrowgpu on the same stream; CUDA events, max over ranks, no host sync"}
        # Greater(int64, 89) -> mask ; Filter ; fused ; Take
        vi = dr  # reuse: regenerate as int64 uniform [0,100)
        N.call("ag_generate_dev", 1, 0x0FF1CE + rank * rows, 0, 99, vi.ptr, rows, None)
        sc = np.array([89], dtype=np.int64)
        mask = DeviceBuffer(rows // 8 + 64)
        ms = timed(lambda: N.call("ag_compare_dev", N.INT64, N.CMP_GT, N.SHAPE_AS, vi.ptr, sc.ctypes.data, mask.ptr, rows, 0, None), W, K)
        others["greater_i64_scalar"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 8.125 * rows / ms / 1e6, "frac": 8.125 * rows / ms / 1e6 / peak, "ms": ms}
        N.call("ag_filter_output_size_dev", mask.ptr, None, 0, rows, 0, scal.ptr, None)
        cnt = int(scal.to_numpy(np.int64, 1)[0])
        sel = cnt / rows
        ms = timed(lambda: N.call("ag_filter_primitive_dev", 64, vi.ptr, None, 0, mask.ptr, None, 0, rows, 0, dout.ptr, None, cnt, scal.ptr + 8, None), W, K)
        fb = (8 + 0.125 + 8 * sel) * rows
        others["filter_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": fb / ms / 1e6, "frac": fb / ms / 1e6 / peak, "ms": ms, "selectivity": sel}
        ms = timed(lambda: N.call("ag_filter_compare_scalar_dev", N.INT64, N.CMP_GT, vi.ptr, sc.ctypes.data, rows, dout.ptr, cnt, scal.ptr + 8, None), W, K)
        fb = (8 + 8 * sel) * rows
        others["fused_greater_filter_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": fb / ms / 1e6, "frac": fb / ms / 1e6 / peak, "ms": ms}
        idx = mask = None
        idx = DeviceBuffer(rows * 4)
        N.call("ag_generate_dev", 2, 0x0FF1CE + 7 + rank * rows, 0, rows - 1, idx.ptr, rows, None)
        bad = DeviceBuffer(64)
        N.call("ag_error_word_reset_dev", bad.ptr, None)
        ms = timed(lambda: N.call("ag_take_primitive_dev", 64, vi.ptr, None, 0, rows, 32, 1, idx.ptr, None, 0, rows, 1, dout.ptr, None, bad.ptr, None), W, K)
        others["take_i64_i32idx_random"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 20.0 * rows / ms / 1e6, "frac": 20.0 * rows / ms / 1e6 / peak, "ms": ms,
                                            "path": "windowed (partition by 16 MB table window -> L2-resident gather -> un-permute), chosen by the on-device probe",
                                            "note": "algorithmic 20 B/row; 100M random int32 indices into a 100M-row int64 table (800 MB); L2 flushed by the 2 GB the call itself moves"}
        N.call("ag_take_set_policy", 1, 0, 0, 0)
        ms = timed(lambda: N.call("ag_take_primitive_dev", 64, vi.ptr, None, 0, rows, 32, 1, idx.ptr, None, 0, rows, 1, dout.ptr, None, bad.ptr, None), 3, max(3, K // 4))
        N.call("ag_take_set_policy", 0, 0, 0, 0)
        others["take_i64_i32idx_random_direct_path"] = {"ms": ms, "frac": 20.0 * rows / ms / 1e6 / peak, "note": "same call forced onto the one-pass gather (round 1's kernel): one DRAM line per gathered row"}
        # sorted indices: the probe keeps the direct kernel, which then streams the table (vector_selection.go:897-911)
        N.call("ag_generate_dev", 5, 0, 0, rows - 1, idx.ptr, rows, None)
        ms = timed(lambda: N.call("ag_take_primitive_dev", 64, vi.ptr, None, 0, rows, 32, 1, idx.ptr, None, 0, rows, 1, dout.ptr, None, bad.ptr, None), W, K)
        others["take_i64_i32idx_sorted"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 20.0 * rows / ms / 1e6, "frac": 20.0 * rows / ms / 1e6 / peak, "ms": ms,
                                            "path": "direct (probe: adjacent indices are neighbours)"}
        N.call("ag_generate_dev", 2, 0x0FF1CE + 7 + rank * rows, 0, rows - 1, idx.ptr, rows, None)
        # Add on sliced operands (Arrow slices are only element-aligned): l.slice(1, n) + r.slice(0, n)
        N.call("ag_generate_dev", 3, 0x94378166 + rank * rows, -(1 << 20), 1 << 20, vi.ptr, rows, None)
        ms = timed(lambda: N.call("ag_arith_binary_dev", N.FLOAT64, N.OP_ADD_CHECKED, N.SHAPE_AA, dl.ptr + 8, vi.ptr, dout.ptr, rows - 1, None), W, K)
        others["add_f64_left_sliced_by_1"] = {"ms": ms, "frac": 24.0 * (rows - 1) / ms / 1e6 / peak, "note": "left operand 8 bytes off a 16-byte boundary: aligned 128-bit loads + shuffle/funnel shift"}
        ms = timed(lambda: N.call("ag_arith_binary_dev", N.FLOAT64, N.OP_ADD_CHECKED, N.SHAPE_AA, dl.ptr + 8, vi.ptr + 8, dout.ptr + 8, rows - 1, None), W, K)
        others["add_f64_all_sliced_by_1"] = {"ms": ms, "frac": 24.0 * (rows - 1) / ms / 1e6 / peak, "note": "all three operands share the misalignment (what executeSpans produces): one head row, then the aligned path"}
        N.call("ag_generate_dev", 1, 0x0FF1CE + rank * rows, 0, 99, vi.ptr, rows, None)
        # rows SURVEY §8(f) marks "next", same device-resident columns: promotion cast, min/max, cumulative sum
        ms = timed(lambda: N.call("ag_cast_numeric_dev", N.INT32, N.INT64, idx.ptr, dout.ptr, rows, None), W, K)
        others["cast_i32_to_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 12.0 * rows / ms / 1e6, "frac": 12.0 * rows / ms / 1e6 / peak, "ms": ms}
        N.call("ag_error_word_reset_dev", bad.ptr, None)
        ms = timed(lambda: N.call("ag_cast_numeric_checked_dev", N.INT64, N.FLOAT64, vi.ptr, None, 0, dout.ptr, rows, 0, 0, bad.ptr, None), W, K)
        others["cast_i64_to_f64_safe"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 16.0 * rows / ms / 1e6, "frac": 16.0 * rows / ms / 1e6 / peak, "ms": ms}
        ms = timed(lambda: N.call("ag_min_max_dev", N.INT64, vi.ptr, rows, scal.ptr, None), W, K)
        others["min_max_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 8.0 * rows / ms / 1e6, "frac": 8.0 * rows / ms / 1e6 / peak, "ms": ms}
        cstate = DeviceBuffer(64)

        def cumsum():
            N.call("ag_cumulative_sum_state_init_dev", cstate.ptr, N.INT64, None, None)
            N.call("ag_cumulative_sum_dev", N.INT64, vi.ptr, None, 0, rows, 0, 0, dout.ptr, None, 0, cstate.ptr, bad.ptr, None)
        ms = timed(cumsum, W, K)
        others["cumulative_sum_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 16.0 * rows / ms / 1e6, "frac": 16.0 * rows / ms / 1e6 / peak, "ms": ms,
                                        "note": "single-pass scan, read once + write once (16 B/row)"}
        vmask = DeviceBuffer(rows // 8 + 64)
        N.call("ag_generate_dev", 4, 0x1234 + rank, 9, 10, vmask.ptr, rows, None)   # 90 % valid
        ovalid = DeviceBuffer(rows // 8 + 64)

        def cumsum_nulls():
            N.call("ag_cumulative_sum_state_init_dev", cstate.ptr, N.INT64, None, None)
            N.call("ag_cumulative_sum_dev", N.INT64, vi.ptr, vmask.ptr, 3, rows, 1, 0, dout.ptr, ovalid.ptr, 0, cstate.ptr, bad.ptr, None)
        ms = timed(cumsum_nulls, W, K)
        others["cumulative_sum_i64_nulls_skip"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 16.25 * rows / ms / 1e6, "frac": 16.25 * rows / ms / 1e6 / peak, "ms": ms,
                                                   "note": "10 % nulls, skip_nulls: the general scan kernel (block-synchronous look-back) + validity pass"}
        # shift_left (checked), bit_wise_xor, divide (checked float NotNull kernel) on resident columns.  vi IS dr (int64 in
        # [0, 100)); dout gets the shift amounts, dl takes the integer results and is regenerated afterwards
        N.call("ag_generate_dev", 1, 0x51F7 + rank, 0, 62, dout.ptr, rows, None)
        N.call("ag_error_word_reset_dev", bad.ptr, None)
        ms = timed(lambda: N.call("ag_arith_checked_dev", N.INT64, N.OP_SHIFT_LEFT_CHECKED, N.SHAPE_AA, vi.ptr, None, 0, dout.ptr, None, 0, dl.ptr, rows, bad.ptr, None), W, K)
        others["shift_left_i64_checked"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 24.0 * rows / ms / 1e6, "frac": 24.0 * rows / ms / 1e6 / peak, "ms": ms}
        ms = timed(lambda: N.call("ag_arith_binary_dev", N.INT64, N.OP_BIT_XOR, N.SHAPE_AA, vi.ptr, dout.ptr, dl.ptr, rows, None), W, K)
        others["bit_wise_xor_i64"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 24.0 * rows / ms / 1e6, "frac": 24.0 * rows / ms / 1e6 / peak, "ms": ms}
        N.call("ag_generate_dev", 3, 0x94378165 + rank * rows, -(1 << 20), 1 << 20, dl.ptr, rows, None)
        N.call("ag_generate_dev", 3, 0x0D1F + rank * rows, 1, 1 << 20, dout.ptr, rows, None)       # divisors >= 1: no error raised
        ms = timed(lambda: N.call("ag_arith_checked_dev", N.FLOAT64, N.OP_DIV_CHECKED, N.SHAPE_AA, dl.ptr, None, 0, dout.ptr, None, 0, dr.ptr, rows, bad.ptr, None), W, K)
        others["divide_f64_checked"] = {"rows_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 24.0 * rows / ms / 1e6, "frac": 24.0 * rows / ms / 1e6 / peak, "ms": ms,
                                        "note": "ScalarBinaryNotNull float kernel with the zero-divisor test per valid slot"}
        # Parquet decode primitives (SURVEY 8f rank 4): bit-unpack 100M 13-bit values, bytes -> bools, def levels -> validity
        nb = 13
        unp = C.c_int64()
        ms = timed(lambda: N.call("ag_parquet_unpack32_dev", vi.ptr, dout.ptr, rows, nb, C.byref(unp), None), W, K)
        ub = rows * nb / 8.0 + rows * 4.0
        others["parquet_unpack32_13bit"] = {"values_per_s": world * rows / ms * 1e3, "gbs_per_gpu": ub / ms / 1e6, "frac": ub / ms / 1e6 / peak, "ms": ms,
                                            "note": "13/8 B in + 4 B out per value"}
        ms = timed(lambda: N.call("ag_parquet_bytes_to_bools_dev", vi.ptr, rows // 8, dout.ptr, rows, None), W, K)
        others["parquet_bytes_to_bools"] = {"values_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 1.125 * rows / ms / 1e6, "frac": 1.125 * rows / ms / 1e6 / peak, "ms": ms,
                                            "note": "1/8 B in + 1 B out per value"}
        N.call("ag_generate_dev", 2, 0xDEF + rank, 0, 1, dr.ptr, rows, None)   # int32 lanes -> int16 levels in {0, 1} pairs
        counts = DeviceBuffer(64)
        ms = timed(lambda: N.call("ag_parquet_def_levels_to_bitmap_dev", dr.ptr, rows, 1, -1, ovalid.ptr, 0, rows, counts.ptr, None), W, K)
        others["parquet_def_levels_to_bitmap"] = {"values_per_s": world * rows / ms * 1e3, "gbs_per_gpu": 2.125 * rows / ms / 1e6, "frac": 2.125 * rows / ms / 1e6 / peak, "ms": ms,
                                                  "note": "flat column: 2 B level in + 1 bit out per value (levels_gt_kernel: 8 levels per 128-bit load, + popcount)"}
        counts.free(); vmask.free(); ovalid.free()
        N.call("ag_generate_dev", 3, 0x94378166 + rank * rows, -(1 << 20), 1 << 20, dr.ptr, rows, None)
        # SURVEY 8f rank 3, same columns: sort_indices (stable radix sort), is_in (1000-value set), unique (100 distinct values)
        N.call("ag_generate_dev", 1, 0x5027 + rank * rows, -(1 << 31), (1 << 31) - 1, vi.ptr, rows, None)
        nn, na = C.c_int64(), C.c_int64()
        ms = timed(lambda: N.call("ag_sort_indices_dev", N.INT64, vi.ptr, None, 0, rows, 0, 0, dout.ptr, C.byref(nn), C.byref(na), None), 1, 3)
        others["sort_indices_i64"] = {"rows_per_s": world * rows / ms * 1e3, "ms": ms, "gbs_per_gpu": 16.0 * rows / ms / 1e6, "frac": 16.0 * rows / ms / 1e6 / peak,
                                      "note": "keys uniform in [-2^31, 2^31): sorted as (key - min), 32 significant bits -> 4 digit passes, the first straight from the column (no NaN/null rows: no class pass), the last writing the uint64 indices; algorithmic 8 B key in + 8 B index out per row; one host sync inside (40 B of statistics)"}
        N.call("ag_generate_dev", 1, 0x15 + rank * rows, 0, 99_999, vi.ptr, rows, None)
        sset = DeviceBuffer(8000)
        hs = np.arange(0, 100_000, 100, dtype=np.int64)
        N.call("ag_upload", sset.ptr, hs.ctypes.data, 8000, None)
        bm1, bm2 = DeviceBuffer(rows // 8 + 64), DeviceBuffer(rows // 8 + 64)
        ms = timed(lambda: N.call("ag_is_in_dev", 64, vi.ptr, None, 0, rows, sset.ptr, None, 0, 1000, 0, bm1.ptr, bm2.ptr, scal.ptr, None), W, K)
        others["is_in_i64_1000_values"] = {"rows_per_s": world * rows / ms * 1e3, "ms": ms, "gbs_per_gpu": 8.25 * rows / ms / 1e6, "frac": 8.25 * rows / ms / 1e6 / peak,
                                           "note": "8 B value in + 2 bitmap bits out per row; the 1000-value set is probed in shared memory (4096 key slots, load factor 1/4, two slots per 128-bit read)"}
        N.call("ag_generate_dev", 1, 0x16 + rank * rows, 0, 99, vi.ptr, rows, None)
        ms = timed(lambda: N.call("ag_unique_dev", 64, vi.ptr, None, 0, rows, dout.ptr, None, rows, scal.ptr, None), 1, 3)
        others["unique_i64_100_distinct"] = {"rows_per_s": world * rows / ms * 1e3, "ms": ms,
                                             "gbs_per_gpu": 8.0 * rows / ms / 1e6, "frac": 8.0 * rows / ms / 1e6 / peak,
                                             "note": "insert (atomicCAS / atomicMin first row) + mark + compaction, 8 B/row algorithmic; L2-resident 4M-slot table first (the full-size one only after an on-device overflow), per-warp seen-key cache"}
        sset.free(); bm1.free(); bm2.free()
        N.call("ag_generate_dev", 1, 0x0FF1CE + rank * rows, 0, 99, vi.ptr, rows, None)
        cstate.free(); idx.free(); bad.free(); scal.free()

    # ---- BASELINE configs 4 and 5 at their full 1B rows, split over the ranks by ag_shard_range; values asserted ----
    if not args.no_full_configs:
        dl.free(); dr.free(); dout.free()
        others.update(full_size_configs(N, comm, dist, rank, world, peak, timed, DeviceBuffer, args.full_rows))
        dl, dr, dout = DeviceBuffer(rows * 8), DeviceBuffer(rows * 8), DeviceBuffer(rows * 8)
        N.call("ag_generate_dev", 3, 0x94378165 + rank * rows, -(1 << 20), 1 << 20, dl.ptr, rows, None)

    launches_total = N.raw().ag_kernel_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None

    # ---- e2e: HOST buffers through the C ABI, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        e_rows = rows
        ha, hb, ho = PinnedArray(e_rows, np.float64), PinnedArray(e_rows, np.float64), PinnedArray(e_rows, np.float64)
        N.call("ag_download", ha.ptr, dl.ptr, e_rows * 8, None)
        N.call("ag_generate_dev", 3, 0x94378166 + rank * rows, -(1 << 20), 1 << 20, dr.ptr, rows, None)
        N.call("ag_download", hb.ptr, dr.ptr, e_rows * 8, None)
        N.call("ag_stream_sync", None)

        htable = N.span_table([(ha.ptr + 8 * pos, hb.ptr + 8 * pos, ho.ptr + 8 * pos, ln) for pos, ln in spans])

        def e2e_step():
            N.call("ag_arith_binary_spans", N.FLOAT64, N.OP_ADD_CHECKED, N.SHAPE_AA, htable, len(spans))
        ke = max(3, min(K, 10))
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            e2e_step()
        dt = max_over_ranks(time.perf_counter() - t0)
        barrier()
        assert np.array_equal(ho.array[:4096], ha.array[:4096] + hb.array[:4096])
        link = link_peaks(N, ha, ho, dl, dout, e_rows * 8, Event, barrier, max_over_ranks)
        e2e = {"value": world * e_rows * ke / dt, "unit": "rows/s", "h2d_bytes_per_step": 16 * e_rows, "d2h_bytes_per_step": 8 * e_rows,
               "ms_per_step": dt / ke * 1e3, "link_gbs": 24.0 * e_rows * ke / dt / 1e9, "link_peak": link,
               "frac_of_link_peak": (24.0 * e_rows * ke / dt / 1e9) / link["bidirectional_gbs"] if link.get("bidirectional_gbs") else None,
               "how": "ag_arith_binary_spans(host ptrs) over the same 200-span chunked layout on ag_host_alloc (pinned) buffers; synchronous API timed by wall clock, max over ranks; "
                      "link_peak = pinned cudaMemcpyAsync of 800 MB each way measured in this run (per GPU, all ranks copying at once)"}
        e2e["config3_upload_once_pipeline"] = c3_pipeline(N, ha, ho, dl, dout, e_rows, rank, Event, barrier, max_over_ranks)
        ha.free(); hb.free(); ho.free()

    # ---- CPU baseline (rank 0, N=1 only) ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = CpuAdd(rows)
        one, one_best, _ = cpu.one_core(2, 5)
        allc, T = cpu.all_cores(1, 3)
        cpu_baseline = {"value": one, "unit": "rows/s", "cores": 1, "kind": cpu.kind, "isa": cpu.isa, "best_step": one_best,
                        "sample": f"the full workload ({rows} rows, 200 spans) x 5 steps through the reference's arithmetic_binary_{cpu.isa}, C harness pinned to one core "
                                  "(1 goroutine per CallFunction, exec.go:164-170)",
                        "all_cores": {"value": allc, "unit": "rows/s", "cores": T, "note": "row-range sharded over all host cores, one pinned thread each; not a reference feature"}}
        del cpu

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_chunked,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "impl": "ours", "config": bench_config(rows, world),
            "detail": {"contiguous_ms_per_step": ms_contig, "per_span_launch_ms_per_step": ms_per_span,
                       "timing": "CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic_bytes(),
                         "traffic_note": "bytes per launch, dram__bytes_read+write from profiles/r2/ncu_full_bench_kernels.csv (ncu --set full of this command's Add kernel)",
                         "peak_kind": peak_kind, "algorithmic_bytes_per_row": 24, "kernel": "binary_spans_kernel<double,OpAdd,AA>",
                         "contiguous_frac": 24.0 * rows / (ms_contig * 1e-3) / 1e9 / peak},
            "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches_timed), "gpu_launches_total": int(launches_total),
            "clocks": clocks, "others": others,
        }
        _emit(line)
    if dist is not None:
        dist.destroy_process_group()


def _emit(line):
    """The ONE JSON line, on the process's original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def _claim_stdout():
    """Everything any library prints (NCCL's version banner, torch notices) goes to stderr: file
    descriptor 1 is pointed at stderr for the whole run and only _emit() writes to the real stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


if __name__ == "__main__":
    main()
