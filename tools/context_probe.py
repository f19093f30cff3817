#!/usr/bin/env python3
"""Cost of context lines (grep -A/-B/-C) on one GPU, device-resident input.

Inputs: 2 GiB of BASELINE configs[1] text (C2 patterns over synthetic syslog, one segment) and 1 GiB of a line-dense text
(lines under 16 bytes).  Cases per input, each on the fast path and on the general path (GPUGREP_FORCE_GENERAL), warmed up
once and then timed --reps times (median of CUDA-event gpu_ms and of wall time): the normal scan with records, the inverted
scan with records, context -C2, context -C100 and -v -C2.  Records go to gpugrep_discard_results (full host delivery, no
Python frame); one more run with a counting callback gives the record count.  Parity: on an 8 MiB head of each input, the
(id, line number) records of -C2 and -v -C2 equal the context model over the oracle's normal scan.  Prints the card name
and power limit (nvidia-smi, read-only query) in the same run; --json PATH also writes the report there.
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

from gpu_api import Stats, marshal  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402
from oracle_api import CALLBACK, load_oracle  # noqa: E402
from test_context_lines import CONTEXT_ID, context_model  # noqa: E402

parser = argparse.ArgumentParser()
parser.add_argument("--c2-mib", type=int, default=2048)
parser.add_argument("--dense-mib", type=int, default=1024)
parser.add_argument("--reps", type=int, default=3)
parser.add_argument("--json", default="", help="also write the report to this file")
args = parser.parse_args()

lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
lib.gpugrep_context_scan_buffer.restype = ctypes.c_int
lib.gpugrep_context_scan_buffer.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                            ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint,
                                            ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
DISCARD = ctypes.cast(lib.gpugrep_discard_results, ctypes.c_void_p)
# (before, after, invert): A = B = 0 is the normal or the inverted scan itself (the entry point runs no context stage then)
CASES = {"records": (0, 0, False), "invert_records": (0, 0, True), "context_C2": (2, 2, False), "context_C100": (100, 100, False),
         "invert_context_C2": (2, 2, True)}


def c2_text(size):
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(host.numpy(), seed=1234)
    return host


def dense_text(size):
    """Lines of 0-11 bytes, the input of tools/invert_probe.py: an 8 MiB seeded sample tiled to `size`."""
    rng = np.random.default_rng(7)
    words = [b"ok", b"a1", b"ERROR", b"zz9", b"port 80", b"", b"\tq", b"GET /x", b"abcdefghij", b"12:34", b"WARN"]
    weights = np.array([10, 10, 10, 10, 1, 10, 10, 10, 10, 10, 10], dtype=float)   # "port 80" (a C2 match) on ~1% of the lines
    picks = rng.choice(len(words), size=(8 << 20) // 5, p=weights / weights.sum())
    sample = b"\n".join(words[k] for k in picks) + b"\n"
    sample = np.frombuffer(sample[: sample.rfind(b"\n", 0, 8 << 20) + 1], dtype=np.uint8)
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    view = host.numpy()
    view[:] = np.tile(sample, -(-size // sample.size))[:size]
    view[-1] = 10
    return host


def context(ptr, size, patterns, before, after, invert, callback=DISCARD):
    pa, fa, ia, n = marshal(patterns)
    st = Stats()
    rc = lib.gpugrep_context_scan_buffer(ptr, size, 1, pa, fa, ia, n, callback, 262140, 4096, 0, before, after, int(invert), None,
                                         ctypes.byref(st))
    assert rc == 0, rc
    return st


def record_count(ptr, size, patterns, before, after, invert):
    total = [0]

    def cb(_results, count):
        total[0] += count

    ccb = CALLBACK(cb)
    context(ptr, size, patterns, before, after, invert, ctypes.cast(ccb, ctypes.c_void_p))
    return total[0]


def parity(host, patterns, head=8 << 20):
    """-C2 and -v -C2 records on the head of the input == the context model over the oracle's normal scan."""
    view = host.numpy()
    cut = int(np.flatnonzero(view[:head] == 10)[-1]) + 1
    text = bytes(view[:cut])
    dev = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    oracle = load_oracle()
    pa, fa, ia, n = marshal(patterns)
    cap = text.count(b"\n") + 1
    out = (ctypes.c_ulonglong * cap)()
    matches, lines = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
    rc = oracle.oracle_lines_buffer(text, ctypes.c_size_t(len(text)), pa, fa, ia, n, 262140, out, ctypes.c_ulonglong(cap),
                                    ctypes.byref(matches), ctypes.byref(lines))
    assert rc == 0
    selected = np.zeros(lines.value, dtype=bool)
    selected[[out[k] for k in range(min(matches.value, cap))]] = True
    ok = True
    for invert in (False, True):
        got = []

        def cb(results, count):
            got.extend((results[k].id, results[k].line_number) for k in range(count))

        ccb = CALLBACK(cb)
        context(dev.data_ptr(), len(text), patterns, 2, 2, invert, ctypes.cast(ccb, ctypes.c_void_p))
        want_lines, is_context = context_model(~selected if invert else selected, 2, 2)
        ok = ok and got == [(CONTEXT_ID if c else 0, int(ln)) for ln, c in zip(want_lines, is_context)]
    return ok


def timed(fn, reps):
    fn()   # warm-up
    runs = [fn() for _ in range(reps)]
    st = runs[len(runs) // 2]
    ms = statistics.median(r.gpu_ms for r in runs)
    return {"gpu_ms": round(ms, 3), "wall_ms": round(statistics.median(r.wall_ms for r in runs), 3), "launches": st.launches,
            "lines": st.lines, "selected": st.matches, "path": st.path, "d2h_bytes": st.d2h_bytes}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60, check=False).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return f"{torch.cuda.get_device_name(0)}, power limit unknown"


def main():
    conditions = card()
    print(f"card: {conditions}")
    report = {"card": conditions, "inputs": {}}
    for label, make, size, patterns in (("c2_syslog", c2_text, args.c2_mib << 20, synth.C2_PATTERNS),
                                        ("dense_short_lines", dense_text, args.dense_mib << 20, synth.C2_PATTERNS)):
        host = make(size)
        ok = parity(host, patterns)
        dev = host.cuda()
        torch.cuda.synchronize()
        ptr = dev.data_ptr()
        cases = {}
        for general in (False, True):
            if general:
                os.environ["GPUGREP_FORCE_GENERAL"] = "1"
            try:
                for case, (before, after, invert) in CASES.items():
                    r = timed(lambda: context(ptr, size, patterns, before, after, invert), args.reps)   # pylint: disable=cell-var-from-loop
                    r["records"] = record_count(ptr, size, patterns, before, after, invert)
                    cases[case + ("_general" if general else "")] = r
            finally:
                os.environ.pop("GPUGREP_FORCE_GENERAL", None)
        report["inputs"][label] = {"bytes": size, "parity": ok, "cases": cases}
        print(f"{label}: {size >> 20} MiB, parity {str(ok).lower()}")
        for case, r in cases.items():
            print(f"  {case:26s} gpu_ms={r['gpu_ms']:9.3f} wall_ms={r['wall_ms']:9.3f} launches={r['launches']:3d} path={r['path']} "
                  f"lines={r['lines']} selected={r['selected']} records={r['records']}")
        del dev, host
        torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w", encoding="utf-8") as handle:
            json.dump(report, handle, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
