#!/usr/bin/env python
"""dictionary_encode on device-resident columns (CUDA events, warm-up first): time, rows/s, algorithmic bytes
(w + 4 per row: read the value, write its index) and their fraction of the HBM copy rate ag_copy_dev reaches in the
same run; unique on the same columns for comparison; per-pass kernel times from a torch.profiler run of its own.

    python scripts/dictionary_encode_bench.py [--out result.json] [--reps 10]

The 100M-row columns (800 / 400 MB) are far larger than L2, so every timed pass reads HBM; the 6M-row column (48 MB)
fits L2 and exists to force the full-size table (3M distinct values overflow the 4M-slot first table).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from arrow_go_b200 import _native as N
from arrow_go_b200.device import DeviceBuffer, Event

CASES = [  # (name, bit width, rows, distinct values)
    ("int64_100m_card100", 64, 100_000_000, 100),
    ("int64_100m_card1m", 64, 100_000_000, 1_000_000),
    ("int32_100m_card100", 32, 100_000_000, 100),
    ("int64_6m_card3m", 64, 6_000_000, 3_000_000),
]
PASS_KERNELS = ("hash_insert_kernel", "table_clear_kernel", "unique_mark_kernel", "dict_rank_count_kernel", "dict_rank_scan_kernel",
                "dict_finalize_kernel", "dict_encode_kernel")


def timed(fn, reps):
    for _ in range(2):
        fn()
    N.call("ag_stream_sync", None)
    times = []
    for _ in range(reps):
        e0, e1 = Event(), Event()
        e0.record(); fn(); e1.record(); e1.sync()
        times.append(e0.elapsed_ms(e1))
    times.sort()
    return {"median_ms": times[len(times) // 2], "min_ms": times[0], "max_ms": times[-1]}


def card_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001 - the numbers are still worth writing
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    N.call("ag_init", 0)
    n_max = max(c[2] for c in CASES)
    vals, idx, dict_out, uniq = DeviceBuffer(n_max * 8 + 64), DeviceBuffer(n_max * 4 + 64), DeviceBuffer(n_max * 8 + 64), DeviceBuffer(n_max * 8 + 64)
    counts, ulen = DeviceBuffer(64), DeviceBuffer(64)

    # HBM copy rate of this card in this run: 800 MB D2D, read + write counted
    copy_bytes = n_max * 8
    cp = timed(lambda: N.call("ag_copy_dev", dict_out.ptr, vals.ptr, copy_bytes, None), args.reps)
    copy_rate = 2 * copy_bytes / (cp["median_ms"] * 1e-3)

    result = {"card": card_info(), "copy": {"bytes_moved": 2 * copy_bytes, **cp, "bytes_per_s": copy_rate}, "cases": []}
    for name, bw, n, card in CASES:
        kind = 1 if bw == 64 else 2
        N.call("ag_generate_dev", kind, 0xD1C7, 0, card - 1, vals.ptr, n, None)
        enc = lambda: N.call("ag_dictionary_encode_dev", bw, vals.ptr, None, 0, n, 0, idx.ptr, None, dict_out.ptr, None, n, counts.ptr, None)
        unq = lambda: N.call("ag_unique_dev", bw, vals.ptr, None, 0, n, uniq.ptr, None, n, ulen.ptr, None)
        te = timed(enc, args.reps)
        tu = timed(unq, args.reps)
        N.call("ag_stream_sync", None)
        k = int(counts.to_numpy("int64", 2)[0])
        alg_bytes = n * (bw // 8 + 4)
        sec = te["median_ms"] * 1e-3
        result["cases"].append({
            "case": name, "rows": n, "bit_width": bw, "distinct": k, "dictionary_encode": te, "unique": tu,
            "rows_per_s": n / sec, "algorithmic_bytes": alg_bytes, "algorithmic_bytes_per_s": alg_bytes / sec,
            "fraction_of_copy_rate": alg_bytes / sec / copy_rate, "ratio_to_unique": te["median_ms"] / tu["median_ms"],
        })
        print(f"{name:22s} dictionary_encode {te['median_ms']:8.3f} ms  unique {tu['median_ms']:8.3f} ms  "
              f"{n / sec / 1e9:6.2f} G rows/s  {alg_bytes / sec / 1e12:5.2f} TB/s alg = {alg_bytes / sec / copy_rate:5.1%} of copy", flush=True)

    if not args.no_profile:
        try:
            result["per_pass_us"] = per_pass(vals, idx, dict_out, counts)
        except Exception as e:  # noqa: BLE001 - the timings above stand without the breakdown
            result["per_pass_us"] = f"profiler failed: {e}"
        print(result["per_pass_us"], flush=True)

    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


def per_pass(vals, idx, dict_out, counts):
    """Device time per kernel of one dictionary_encode call (mean of 3), from a torch.profiler trace of its own:
    tracing slows the host, not the kernels."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    passes = {}
    for name, bw, n, card in CASES:
        kind = 1 if bw == 64 else 2
        N.call("ag_generate_dev", kind, 0xD1C7, 0, card - 1, vals.ptr, n, None)
        N.call("ag_stream_sync", None)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                N.call("ag_dictionary_encode_dev", bw, vals.ptr, None, 0, n, 0, idx.ptr, None, dict_out.ptr, None, n, counts.ptr, None)
            N.call("ag_stream_sync", None)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            dev_us = getattr(ev, "device_time", None)
            if dev_us is None:
                dev_us = getattr(ev, "cuda_time", 0.0)
            for kname in PASS_KERNELS:
                if kname in ev.name:
                    per[kname] = per.get(kname, 0.0) + dev_us / 3.0
        passes[name] = {k: round(v, 2) for k, v in per.items()} or "not captured"
    return passes


if __name__ == "__main__":
    main()
