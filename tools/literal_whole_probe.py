"""Whole-word and whole-line fixed strings (gpugrep_literal_whole_scan_buffer, grep -F -w / -F -x) against the plain literal
scan; writes profiles/literal_whole_probe.json.

The setup of tools/literal_probe.py: seeded configs[1] syslog (>= 2 GiB, device-resident) with IOC-shaped lists of 1k, 10k
and 100k literals planted in it: one line in 2,000 gets " ioc=<literal>" (a word), one in 4,000 " x<literal>y" (inside a
longer word: selected by -F only) and one in 6,000 is replaced by the literal alone (a whole line).  Per list, the routes
-F, -Fw and -Fx, each count-only (NULL callback) and with records (a callback that counts them), alternated over --rounds
rounds after one warm-up round; each reports the median and the range of `gpu_ms` (device events around the segment's
kernels), the median wall time, launches, selected lines and path.  At 1k literals also the regex route of -Fw
(every literal as \\xHH inside (?:^|[^0-9A-Za-z_])...(?:[^0-9A-Za-z_]|$), gpugrep_scan_buffer).
Dense reject (synth.dense_reject_bytes, 64 MiB repeated to --dense-gib): every line holds `error` inside longer words and
one in 97 also as a word, so -F selects every line.  With records, -Fw and -F run the same kernels plus the filter, and
their difference per GiB of selected-line bytes is the filter's cost.  Count-only, -Fw also swaps the key emit and
k_count_keys of -F for the record emit (line numbers, NUL scans) and k_dedupe_records: that difference is reported apart,
as the whole extra cost of a count-only -Fw.
Usage:
    python tools/literal_whole_probe.py [--gib 2] [--sizes 1000,10000,100000] [--out profiles/literal_whole_probe.json]
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gpu_api import Stats, marshal  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402
from literal_probe import iocs  # noqa: E402
from oracle_api import CALLBACK  # noqa: E402

_ROUTES = (("F", 0), ("Fw", 1), ("Fx", 2))


def main() -> None:  # pylint: disable=too-many-locals,too-many-statements
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=2.0)
    ap.add_argument("--sizes", default="1000,10000,100000")
    ap.add_argument("--dense-gib", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "literal_whole_probe.json"))
    args = ap.parse_args()
    import torch  # pylint: disable=import-outside-toplevel

    lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
    sel = lib.gpugrep_literal_scan_buffer
    sel.restype = ctypes.c_int
    sel.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int,
                    ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    whole = lib.gpugrep_literal_whole_scan_buffer
    whole.restype = ctypes.c_int
    whole.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_uint, ctypes.c_void_p,
                      ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    reg = lib.gpugrep_scan_buffer
    reg.restype = ctypes.c_int
    reg.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                    ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=False).stdout.strip().splitlines()
    results = {"card": smi[0] if smi else "unknown", "lists": []}
    counted = [0]

    def on_batch(_results, count):
        counted[0] += count

    callback = CALLBACK(on_batch)
    cb = ctypes.cast(callback, ctypes.c_void_p)

    def summary(samples: list[dict]) -> dict:
        ms = sorted(r["gpu_ms"] for r in samples)
        walls = sorted(r["wall_s"] for r in samples)
        out = dict(samples[-1])
        out.update({"gpu_ms": ms[len(ms) // 2], "gpu_ms_min": ms[0], "gpu_ms_max": ms[-1], "wall_s": walls[len(walls) // 2],
                    "rounds": len(samples)})
        return out

    def run(route: str, mode: int, dev, size: int, la, fa, n: int, records: bool, regex=None) -> dict:
        st = Stats()
        counted[0] = 0
        c = cb if records else None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if regex is not None:
            pa, pfa, pia, pn = regex
            rc = reg(dev.data_ptr(), size, 1, pa, pfa, pia, pn, c, 262140, 4096, 0, None, ctypes.byref(st))
        elif mode == 0:
            rc = sel(dev.data_ptr(), size, 1, la, fa, n, c, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(st))
        else:
            rc = whole(dev.data_ptr(), size, 1, la, fa, n, mode, c, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(st))
        wall = time.perf_counter() - t0
        return {"route": route, "records": records, "rc": rc, "gpu_ms": round(st.gpu_ms, 3), "wall_s": round(wall, 4),
                "launches": st.launches, "lines": counted[0] if records else st.matches, "path": st.path}

    base = synth.syslog_bytes(256 << 20, seed=7)
    reps = max(1, int(args.gib * (1 << 30) // len(base)))
    for size in [int(s) for s in args.sizes.split(",")]:
        lits = iocs(size, seed=size)
        lines = base.split(b"\n")
        for k in range(0, len(lines), 2000):
            lit = lits[(k // 2000) % len(lits)]
            lines[k] += b" ioc=" + lit
            if k % 4000 == 0 and k + 1 < len(lines):
                lines[k + 1] += b" x" + lit + b"y"
            if k % 6000 == 0 and k + 2 < len(lines):
                lines[k + 2] = lit
        data = b"\n".join(lines) * reps
        dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        n = len(lits)
        la = (ctypes.c_char_p * n)(*lits)
        fa = (ctypes.c_uint * n)(*([0] * n))
        entry = {"literals": n, "bytes": len(data)}
        t0 = time.perf_counter()   # the first call compiles (and caches) the whole-word / whole-line set
        whole(dev.data_ptr(), 4096, 1, la, fa, n, 1, None, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(Stats()))
        entry["whole_compile_s"] = round(time.perf_counter() - t0, 3)
        sel(dev.data_ptr(), 4096, 1, la, fa, n, None, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(Stats()))
        regex = None
        if n <= 1000:
            pats = ["(?:^|[^0-9A-Za-z_])(?:" + "".join(f"\\x{b:02x}" for b in lit) + ")(?:[^0-9A-Za-z_]|$)" for lit in lits]
            regex = marshal(pats, [8] * n, [0] * n)
        runs: dict = {}
        for round_no in range(args.rounds + 1):   # (round 0 warms up)
            for records in (False, True):
                for route, mode in _ROUTES:
                    r = run(route, mode, dev, len(data), la, fa, n, records)
                    if round_no:
                        runs.setdefault((route, records), []).append(r)
                if regex is not None:
                    r = run("regex_w", 1, dev, len(data), la, fa, n, records, regex)
                    if round_no:
                        runs.setdefault(("regex_w", records), []).append(r)
        entry["runs"] = [summary(r) for r in runs.values()]
        print(json.dumps(entry), flush=True)
        results["lists"].append(entry)
        del dev
        torch.cuda.empty_cache()
    # dense reject: -F selects every line, -Fw one in 97
    block, _ = synth.dense_reject_bytes((64 << 20) // 230, seed=1)
    data = block * max(1, int(args.dense_gib * (1 << 30) // len(block)))
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    la = (ctypes.c_char_p * 1)(b"error")
    fa = (ctypes.c_uint * 1)(0)
    runs = {}
    for round_no in range(args.rounds + 1):
        for records in (False, True):
            for route, mode in _ROUTES[:2]:
                r = run(route, mode, dev, len(data), la, fa, 1, records)
                if round_no:
                    runs.setdefault((route, records), []).append(r)
    runs = {key: summary(r) for key, r in runs.items()}
    dense = {"bytes": len(data), "runs": list(runs.values())}
    gib = len(data) / (1 << 30)   # every line is selected by -F: the filter reads all of them
    dense["filter_ms_per_selected_gib"] = round((runs[("Fw", True)]["gpu_ms"] - runs[("F", True)]["gpu_ms"]) / gib, 3)
    dense["count_only_extra_ms_per_selected_gib"] = round((runs[("Fw", False)]["gpu_ms"] - runs[("F", False)]["gpu_ms"]) / gib, 3)
    print(json.dumps(dense), flush=True)
    results["dense_reject"] = dense
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as handle:
        json.dump(results, handle, indent=1)


if __name__ == "__main__":
    main()
