"""Fixed strings with reports (gpugrep_literal_report_scan_buffer) against the selection-only literal scan and the escaped-regex
route with ids, on IOC-shaped lists; writes profiles/literal_report_probe.json.

The setup of tools/literal_probe.py: seeded configs[1] syslog (>= 2 GiB, device-resident) with one planted IOC per 2,000
lines, lists of 1k, 10k, 100k and ~1M literals, ids = index, every literal SINGLEMATCH.  Per list: host compile time of the
report set, and the wall time of three routes, alternated, each with a callback that counts its records: the selection-only
literal scan (gpugrep_literal_scan_buffer), the report scan, and - where the regex compiler takes the re.escape-d list (up to
--regex-max) - gpugrep_scan_buffer of the escaped set with the same ids.  The second run of each route is the one reported.
Then `grep -F -o` of the 100k list over a 64 MiB file: the automaton-free route of utils.grep, and the route it replaced (the
re.escape-d list as regular expressions), the latter in a subprocess cut off after --before-timeout seconds.  Usage:
    python tools/literal_report_probe.py [--gib 2] [--sizes 1000,10000,100000,1000000] [--out profiles/literal_report_probe.json]
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gpu_api import Stats, marshal  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402
from literal_probe import iocs  # noqa: E402
from oracle_api import CALLBACK  # noqa: E402

_BEFORE = """
import re, sys, time
sys.path.insert(0, {root!r})
from hypergrep_b200 import utils
lits = open({lits!r}).read().split("\\n")
t0 = time.perf_counter()
got, code = utils.grep({path!r}, [re.escape(lit) for lit in lits], only_matching=True)
print(time.perf_counter() - t0, len(got), code)
"""


def main() -> None:  # pylint: disable=too-many-locals,too-many-statements
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=2.0)
    ap.add_argument("--sizes", default="1000,10000,100000,1000000")
    ap.add_argument("--regex-max", type=int, default=10000)
    ap.add_argument("--before-timeout", type=float, default=60.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "literal_report_probe.json"))
    args = ap.parse_args()
    import torch  # pylint: disable=import-outside-toplevel

    lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
    sel = lib.gpugrep_literal_scan_buffer
    sel.restype = ctypes.c_int
    sel.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int,
                    ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    buffer_args = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                   ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
    rep = lib.gpugrep_literal_report_scan_buffer
    rep.restype, rep.argtypes = ctypes.c_int, buffer_args
    reg = lib.gpugrep_scan_buffer
    reg.restype, reg.argtypes = ctypes.c_int, buffer_args
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=False).stdout.strip().splitlines()
    base = synth.syslog_bytes(256 << 20, seed=7)
    reps = max(1, int(args.gib * (1 << 30) // len(base)))
    results = {"card": smi[0] if smi else "unknown", "bytes": len(base) * reps, "lists": []}
    counted = [0]

    def on_batch(_results, count):
        counted[0] += count

    callback = CALLBACK(on_batch)
    cb = ctypes.cast(callback, ctypes.c_void_p)
    for size in [int(s) for s in args.sizes.split(",")]:
        lits = iocs(size, seed=size)
        lines = base.split(b"\n")
        for k in range(0, len(lines), 2000):   # one planted hit per 2,000 lines
            lines[k] += b" ioc=" + lits[(k // 2000) % len(lits)]
        data = b"\n".join(lines) * reps
        dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        n = len(lits)
        la = (ctypes.c_char_p * n)(*lits)
        fa = (ctypes.c_uint * n)(*([8] * n))
        ia = (ctypes.c_uint * n)(*range(n))
        entry = {"literals": n}
        t0 = time.perf_counter()   # the first call compiles (and caches) the report set; 4 KiB of text take no time
        rc = rep(dev.data_ptr(), 4096, 1, la, fa, ia, n, None, 262140, 4096, 0, None, ctypes.byref(Stats()))
        entry["report_compile_s"] = time.perf_counter() - t0
        sel(dev.data_ptr(), 4096, 1, la, fa, n, None, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(Stats()))
        pa = None
        if n <= args.regex_max:
            pa, pfa, pia, pn = marshal(["".join(f"\\x{b:02x}" for b in lit) for lit in lits], [8] * n, list(range(n)))
            t0 = time.perf_counter()
            entry["regex_compile_rc"] = lib.check_patterns(pa, pfa, pia, pn)
            entry["regex_compile_s"] = time.perf_counter() - t0
        runs = {"selection": [], "report": [], "regex": []}
        for _ in range(2):
            for route in ("selection", "report", "regex"):
                if route == "regex" and pa is None:
                    continue
                st = Stats()
                counted[0] = 0
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if route == "selection":
                    rc = sel(dev.data_ptr(), len(data), 1, la, fa, n, cb, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(st))
                elif route == "report":
                    rc = rep(dev.data_ptr(), len(data), 1, la, fa, ia, n, cb, 262140, 4096, 0, None, ctypes.byref(st))
                else:
                    rc = reg(dev.data_ptr(), len(data), 1, pa, pfa, pia, pn, cb, 262140, 4096, 0, None, ctypes.byref(st))
                wall = time.perf_counter() - t0
                runs[route].append({"rc": rc, "wall_s": round(wall, 4), "gbps": round(len(data) / wall / 1e9, 2), "records": counted[0],
                                    "gpu_ms": round(st.gpu_ms, 2), "path": st.path, "launches": st.launches})
        entry.update({route: r[-1] for route, r in runs.items() if r})
        if runs["regex"]:
            entry["same_records_as_regex"] = runs["report"][-1]["records"] == runs["regex"][-1]["records"]
        print(json.dumps(entry), flush=True)
        results["lists"].append(entry)
        del dev
        torch.cuda.empty_cache()
    # grep -F -o with 100k literals over 64 MiB
    lits = [lit.decode() for lit in iocs(100_000, seed=100_000)]
    lines = synth.syslog_bytes(64 << 20, seed=9).split(b"\n")
    for k in range(0, len(lines), 2000):
        lines[k] += b" ioc=" + lits[(k // 2000) % len(lits)].encode() + b" first=" + lits[0].encode()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "g.log")
        with open(path, "wb") as handle:
            handle.write(b"\n".join(lines))
        lits_path = os.path.join(tmp, "lits.txt")
        with open(lits_path, "w", encoding="utf-8") as handle:
            handle.write("\n".join(lits))
        grep_res = {"literals": len(lits), "bytes": os.path.getsize(path)}
        for _ in range(2):
            t0 = time.perf_counter()
            got, code = utils.grep(path, lits, fixed_strings=True, only_matching=True)
            grep_res["after_wall_s"] = round(time.perf_counter() - t0, 3)
            grep_res["after_parts"] = len(got)
            grep_res["after_rc"] = code
        try:
            proc = subprocess.run([sys.executable, "-c", _BEFORE.format(root=ROOT, lits=lits_path, path=path)], capture_output=True, text=True,
                                  timeout=args.before_timeout, check=False)
            wall, parts, code = proc.stdout.split()
            grep_res.update({"before_wall_s": round(float(wall), 3), "before_parts": int(parts), "before_rc": int(code)})
        except subprocess.TimeoutExpired:
            grep_res["before_wall_s"] = f"not finished after {args.before_timeout:.0f} s"
    print(json.dumps(grep_res), flush=True)
    results["grep_only_matching_100k"] = grep_res
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as handle:
        json.dump(results, handle, indent=1)


if __name__ == "__main__":
    main()
