#!/usr/bin/env python3
"""Cost of count-only scans against scans with records on one GPU, device-resident input, one segment per call.

Inputs (BASELINE shapes): 2 GiB of configs[1] syslog text with the C2 set (32 patterns) and with the C1 set ("ERROR"); 2 GiB
of planted syslog text with the C3 set (1,000 IOC patterns); 1 GiB of configs[4] JSON-ish text (2-16 KiB lines) with
10,000 caseless patterns; and the configs[1] text with a NUL in every 1,000th line (C2 set).  Per input, each case is
warmed up once and then timed --reps times (median of CUDA-event gpu_ms over all kernels of the call, and of the
streaming kernel alone): count-only (NULL callback) and with records (gpugrep_discard_results as the callback: records
copied and delivered, no Python frame).  gpu_ms is also given per 2 GiB.  --profile adds a torch.profiler pass per input
with the kernel times of one call of each case.  Prints the card name and power limit; --json PATH also writes the
report there.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gpu_api import scan_buffer  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402

parser = argparse.ArgumentParser()
parser.add_argument("--mib", type=int, default=2048, help="size of the syslog inputs (the configs[4] input is half of it)")
parser.add_argument("--reps", type=int, default=5)
parser.add_argument("--only", default="", help="comma-separated input names")
parser.add_argument("--profile", action="store_true", help="per-kernel times from torch.profiler (a separate pass)")
parser.add_argument("--label", default="", help="name of the build measured (e.g. before / after), stored in the report")
parser.add_argument("--json", default="", help="also write the report to this file")
args = parser.parse_args()

lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
DISCARD = ctypes.cast(lib.gpugrep_discard_results, ctypes.c_void_p).value


def syslog(size, seed=1234, plants=None, plant_ppm=0):
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(host.numpy(), seed=seed, plants=plants, plant_ppm=plant_ppm)
    return host


def with_nuls(size):
    host = syslog(size)
    view = host.numpy()
    nl = np.flatnonzero(view == 10)[::1000]
    view[nl[nl + 20 < size] + 20] = 0   # byte 20 of every 1,000th line
    return host


def jsonish(size):
    sample = np.frombuffer(synth.jsonish_bytes(8 << 20, patterns_to_plant=["session_4242 failed", "code=E31337abcd"]), dtype=np.uint8)
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    host.numpy()[:] = np.tile(sample, -(-size // sample.size))[:size]
    host[-1] = 10
    return host


def inputs():
    size = args.mib << 20
    c3, plants = synth.c3_patterns()
    c5 = synth.c5_patterns(10000)
    yield "c2_syslog", lambda: syslog(size), synth.C2_PATTERNS, None
    yield "c1_syslog", lambda: syslog(size), synth.C1_PATTERNS, None
    yield "c3_ioc", lambda: syslog(size, seed=4321, plants=plants, plant_ppm=1000), c3, None
    yield "c5_long_lines", lambda: jsonish(size // 2), c5, [15] * len(c5)
    yield "c2_with_nuls", lambda: with_nuls(size), synth.C2_PATTERNS, None


def call(ptr, size, patterns, flags, records):
    if records:
        # the records path with the native discard callback (scan_buffer's own Python callback would dominate)
        from gpu_api import Stats, marshal  # pylint: disable=import-outside-toplevel

        pa, fa, ia, n = marshal(patterns, flags)
        st = Stats()
        rc = lib.gpugrep_scan_buffer(ptr, size, 1, pa, fa, ia, n, DISCARD, 262140, 4096, 0, None, ctypes.byref(st))
    else:
        rc, _, st = scan_buffer(lib, ptr, size, 1, patterns, flags, collect=False)
    assert rc == 0, rc
    return st


def timed(fn, reps, size):
    fn()
    runs = [fn() for _ in range(reps)]
    ms = statistics.median(r.gpu_ms for r in runs)
    st = runs[-1]
    return {"gpu_ms": round(ms, 4), "gpu_ms_per_2GiB": round(ms * (2 << 30) / size, 4),
            "gpu_ms_all": [round(r.gpu_ms, 4) for r in runs],
            "stream_ms": round(statistics.median(r.stream_kernel_ms for r in runs), 4),
            "launches": st.launches, "path": st.path, "matches": st.matches, "lines": st.lines, "candidates": st.candidates,
            "nul_segments": st.reserved}


def kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile  # pylint: disable=import-outside-toplevel

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = defaultdict(float)
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
            name = ev.name.split("(")[0].split("<")[0].replace("void ", "").replace("gpugrep::", "")
            out[name] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    return {k: round(v, 1) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60, check=False).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "unknown"
    return name, q


def main():
    name, limits = card()
    print(f"card: {name}, power limit / max SM clock {limits}")
    lib.gpugrep_scan_buffer.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                                        ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
    report = {"card": name, "power_limit_max_sm_clock": limits, "build": args.label, "inputs": {}}
    only = set(filter(None, args.only.split(",")))
    for label, make, patterns, flags in inputs():
        if only and label not in only:
            continue
        host = make()
        size = host.numel()
        dev = host.cuda()
        del host
        torch.cuda.synchronize()
        ptr = dev.data_ptr()
        cases = {"count_only": timed(lambda: call(ptr, size, patterns, flags, False), args.reps, size),
                 "records": timed(lambda: call(ptr, size, patterns, flags, True), args.reps, size)}
        assert cases["count_only"]["matches"] == cases["records"]["matches"], label
        entry = {"bytes": size, "cases": cases}
        if args.profile:
            entry["kernels_us"] = {case: kernel_times(lambda records=(case == "records"): call(ptr, size, patterns, flags, records))
                                   for case in ("count_only", "records")}
        report["inputs"][label] = entry
        print(f"{label}: {size >> 20} MiB")
        for case, r in cases.items():
            print(f"  {case:10s} gpu_ms={r['gpu_ms']:9.4f} per2GiB={r['gpu_ms_per_2GiB']:9.4f} stream_ms={r['stream_ms']:8.4f} "
                  f"launches={r['launches']} path={r['path']} matches={r['matches']} nul_segments={r['nul_segments']}")
        if args.profile:
            for case, ks in entry["kernels_us"].items():
                print(f"  {case} kernels (us): " + ", ".join(f"{k} {v}" for k, v in ks.items()))
        del dev
        torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w", encoding="utf-8") as handle:
            json.dump(report, handle, indent=1)


if __name__ == "__main__":
    main()
