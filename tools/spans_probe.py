#!/usr/bin/env python3
"""Cost of `grep -o` on the span route (gpugrep_match_spans) against the reference route (re.finditer per matched line), one GPU.

Input: --mib MiB of BASELINE configs[1] text (synthetic syslog) in a file, with a planted string that holds a match of every
probe pattern on --plant-ppm of the lines (default 900,000: over 1M matched lines per pattern in 256 MiB).  For each probe pattern: wall time of
utils.grep(only_matching=True) on the span route (variable-width patterns) or the match-end route (the fixed-width one), and
on the reference route (utils._span_widths patched to None), median of --reps runs, with the outputs compared; then one
gpugrep_match_spans call over the pattern's matched lines (the text grep hands to it) with its CUDA-event gpu_ms and wall
time, median of --reps after a warm-up.  Prints the card name and power limit (nvidia-smi, read-only query) in the same run;
--json PATH also writes the report there.
"""
import argparse
import ctypes
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gpu_api import Stats  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402

PATTERNS = [r"port [0-9]+", r"user=\w+", r"rhost=10\.[0-9]+\.[0-9]+\.[0-9]+", r"ERROR.*", r"id=[0-9a-f]{12}"]

parser = argparse.ArgumentParser()
parser.add_argument("--mib", type=int, default=256)
parser.add_argument("--plant-ppm", type=int, default=900_000)
parser.add_argument("--reps", type=int, default=3)
parser.add_argument("--json", default="", help="also write the report to this file")
args = parser.parse_args()


class Span(ctypes.Structure):
    _fields_ = [("line_number", ctypes.c_ulonglong), ("start", ctypes.c_uint), ("end", ctypes.c_uint)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60, check=False).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return f"{torch.cuda.get_device_name(0)}, power limit unknown"


def timed(fn, reps):
    times, result = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        result = fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), result


def main():
    conditions = card()
    print(f"card: {conditions}")
    lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
    lib.gpugrep_set_device(0)
    entry = lib.gpugrep_match_spans
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                      ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
    text = np.empty(args.mib << 20, dtype=np.uint8)
    plants = [f"port {p} user={u} rhost=10.{a}.{b}.{c} id={h:012x} ERROR {m}"
              for p, u, a, b, c, h, m in zip([22, 443, 8080, 31337], ["root", "alice", "svc_backup", "x"], [0, 1, 12, 255],
                                             [4, 40, 200, 9], [7, 77, 1, 250], [0xdeadbeef01, 0xa1, 0xfffffffffff, 0x42],
                                             ["disk quota", "timeout", "auth failed", "retry"])]
    synth.fill_syslog(text, seed=1234, plants=plants, plant_ppm=args.plant_ppm)
    data = text.tobytes()
    lines = data.splitlines(keepends=True)
    report = {"card": conditions, "text_mib": args.mib, "plant_ppm": args.plant_ppm, "lines": len(lines), "reps": args.reps,
              "patterns": []}
    with tempfile.NamedTemporaryFile(suffix=".log") as handle:
        handle.write(data)
        handle.flush()
        utils.grep(handle.name, ["port [0-9]+"], only_matching=True)   # warm-up: CUDA context, slots
        for pattern in PATTERNS:
            width = utils._span_widths([pattern])[0]  # pylint: disable=protected-access
            exact = utils._span_exact([pattern])[0]  # pylint: disable=protected-access
            route_s, (got, _) = timed(lambda p=pattern: utils.grep(handle.name, [p], only_matching=True), args.reps)
            original = utils._span_widths  # pylint: disable=protected-access
            utils._span_widths = lambda _patterns: None  # pylint: disable=protected-access
            try:
                reference_s, (expected, _) = timed(lambda p=pattern: utils.grep(handle.name, [p], only_matching=True), args.reps)
            finally:
                utils._span_widths = original  # pylint: disable=protected-access
            assert got == expected, pattern
            compiled = re.compile(pattern.encode())
            matched = b"".join(line for line in lines if line.endswith(b"\n") and compiled.search(line))
            capacity = 4 * len(got) + 1024
            out = (Span * capacity)()
            found = ctypes.c_size_t(0)
            gpu_ms, call_ms = [], []
            for k in range(args.reps + 1):
                stats = Stats()
                t0 = time.perf_counter()
                rc = entry(matched, len(matched), 0, pattern.encode(), 262140, out, capacity, ctypes.byref(found), ctypes.byref(stats))
                wall = (time.perf_counter() - t0) * 1e3
                assert rc == 0 and found.value == len(got), (pattern, rc, found.value, len(got))
                if k:
                    gpu_ms.append(stats.gpu_ms)
                    call_ms.append(wall)
            row = {"pattern": pattern, "route": "spans" if width <= 0 else "match ends", "width": width, "span_exact": exact,
                   "matched_lines": sum(1 for line in lines if compiled.search(line)), "spans": len(got), "matched_bytes": len(matched),
                   "grep_route_s": round(route_s, 3), "grep_reference_s": round(reference_s, 3),
                   "speedup": round(reference_s / route_s, 2), "span_call_gpu_ms": round(statistics.median(gpu_ms), 3),
                   "span_call_wall_ms": round(statistics.median(call_ms), 3)}
            report["patterns"].append(row)
            print(json.dumps(row))
    if args.json:
        with open(args.json, "w", encoding="utf-8") as out_file:
            json.dump(report, out_file, indent=1)
            out_file.write("\n")


if __name__ == "__main__":
    main()
