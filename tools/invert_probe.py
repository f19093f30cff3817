#!/usr/bin/env python3
"""Cost of inverted matching (grep -v) on one GPU, device-resident input.

Inputs: 2 GiB of BASELINE configs[1] text (C2 patterns over synthetic syslog, one segment) and 1 GiB of a line-dense text
(lines under 16 bytes).  Cases per input, each warmed up once and then timed --reps times (median of CUDA-event gpu_ms):
count-only, inverted count-only, inverted with records (gpugrep_discard_results as the callback: full host delivery, no
Python frame) and the same on the general path (GPUGREP_FORCE_GENERAL).  Parity: on an 8 MiB head of each input, the
inverted line numbers equal the complement of the oracle's normal scan, over the oracle's line count.  Prints the card name
and power limit; --json PATH also writes the report there.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gpu_api import Stats, marshal, scan_buffer  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402
from oracle_api import CALLBACK, load_oracle  # noqa: E402

parser = argparse.ArgumentParser()
parser.add_argument("--c2-mib", type=int, default=2048)
parser.add_argument("--dense-mib", type=int, default=1024)
parser.add_argument("--reps", type=int, default=3)
parser.add_argument("--json", default="", help="also write the report to this file")
args = parser.parse_args()

lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
lib.gpugrep_invert_scan_buffer.restype = ctypes.c_int
lib.gpugrep_invert_scan_buffer.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p,
                                           ctypes.c_void_p]
DISCARD = ctypes.cast(lib.gpugrep_discard_results, ctypes.c_void_p)


def invert(ptr, size, patterns, callback=None):
    pa, fa, ia, n = marshal(patterns)
    st = Stats()
    rc = lib.gpugrep_invert_scan_buffer(ptr, size, 1, pa, fa, ia, n, callback, 262140, 4096, 0, None, ctypes.byref(st))
    assert rc == 0, rc
    return st


def normal_count(ptr, size, patterns):
    rc, _, st = scan_buffer(lib, ptr, size, 1, patterns, collect=False)
    assert rc == 0, rc
    return st


def c2_text(size):
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(host.numpy(), seed=1234)
    return host


def dense_text(size):
    """Lines of 0-11 bytes: an 8 MiB seeded sample tiled to `size` (the sample ends with '\\n')."""
    rng = np.random.default_rng(7)
    words = [b"ok", b"a1", b"ERROR", b"zz9", b"port 80", b"", b"\tq", b"GET /x", b"abcdefghij", b"12:34", b"WARN"]
    weights = np.array([10, 10, 10, 10, 1, 10, 10, 10, 10, 10, 10], dtype=float)   # "port 80" (a C2 match) on ~1% of the lines
    picks = rng.choice(len(words), size=(8 << 20) // 5, p=weights / weights.sum())
    sample = b"\n".join(words[k] for k in picks) + b"\n"
    sample = np.frombuffer(sample[: sample.rfind(b"\n", 0, 8 << 20) + 1], dtype=np.uint8)
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    view = host.numpy()
    reps = -(-size // sample.size)
    view[:] = np.tile(sample, reps)[:size]
    view[-1] = 10
    return host


def parity(host, patterns, head=8 << 20):
    """Inverted line numbers on the head of the input == complement of the oracle's normal scan."""
    view = host.numpy()
    cut = int(np.flatnonzero(view[:head] == 10)[-1]) + 1
    text = bytes(view[:cut])
    dev = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    got = []

    def cb(results, count):
        got.extend(results[k].line_number for k in range(count))

    ccb = CALLBACK(cb)
    st = invert(dev.data_ptr(), len(text), patterns, ctypes.cast(ccb, ctypes.c_void_p))
    oracle = load_oracle()
    pa, fa, ia, n = marshal(patterns)
    cap = st.lines + 1
    out = (ctypes.c_ulonglong * cap)()
    matches, lines = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)

    rc = oracle.oracle_lines_buffer(text, ctypes.c_size_t(len(text)), pa, fa, ia, n, 262140, out, ctypes.c_ulonglong(cap),
                                    ctypes.byref(matches), ctypes.byref(lines))
    assert rc == 0
    matched = {out[k] for k in range(min(matches.value, cap))}
    complement = [k for k in range(lines.value) if k not in matched]
    return got == complement and lines.value == st.lines


def timed(fn, reps):
    fn()   # warm-up
    runs = [fn() for _ in range(reps)]
    st = runs[len(runs) // 2]
    ms = statistics.median(r.gpu_ms for r in runs)
    return {"gpu_ms": round(ms, 3), "wall_ms": round(statistics.median(r.wall_ms for r in runs), 3), "launches": st.launches,
            "lines": st.lines, "matches": st.matches, "path": st.path, "GB_per_s": round(st.bytes_scanned / ms / 1e6, 1)}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                               timeout=60, check=False).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        limit = "unknown"
    return name, limit


def main():
    name, limit = card()
    print(f"card: {name}, power limit {limit}")
    report = {"card": name, "power_limit": limit, "inputs": {}}
    for label, make, size, patterns in (("c2_syslog", c2_text, args.c2_mib << 20, synth.C2_PATTERNS),
                                        ("dense_short_lines", dense_text, args.dense_mib << 20, synth.C2_PATTERNS)):
        host = make(size)
        ok = parity(host, patterns)
        dev = host.cuda()
        torch.cuda.synchronize()
        ptr = dev.data_ptr()
        cases = {
            "count_only": timed(lambda: normal_count(ptr, size, patterns), args.reps),
            "invert_count_only": timed(lambda: invert(ptr, size, patterns), args.reps),
            "invert_records": timed(lambda: invert(ptr, size, patterns, DISCARD), args.reps),
        }
        os.environ["GPUGREP_FORCE_GENERAL"] = "1"
        try:
            cases["invert_records_general"] = timed(lambda: invert(ptr, size, patterns, DISCARD), args.reps)
        finally:
            del os.environ["GPUGREP_FORCE_GENERAL"]
        assert cases["invert_count_only"]["matches"] == cases["count_only"]["lines"] - cases["count_only"]["matches"]
        assert cases["invert_records"]["matches"] == cases["invert_count_only"]["matches"] == cases["invert_records_general"]["matches"]
        report["inputs"][label] = {"bytes": size, "parity": ok, "cases": cases}
        print(f"{label}: {size >> 20} MiB, parity {str(ok).lower()}")
        for case, r in cases.items():
            print(f"  {case:24s} gpu_ms={r['gpu_ms']:9.3f} wall_ms={r['wall_ms']:9.3f} launches={r['launches']:3d} path={r['path']} "
                  f"lines={r['lines']} selected/matched={r['matches']} GB/s={r['GB_per_s']}")
        del dev, host
        torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w", encoding="utf-8") as handle:
            json.dump(report, handle, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
