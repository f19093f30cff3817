"""Per-pattern line counts (gpugrep_pattern_counts_buffer) against the count-only scan and the multi-id route they replace;
writes profiles/pattern_counts_probe.json.

Device-resident configs[1] text (synth.fill_syslog, --gib GiB) with these sets:
 - configs[2]: the 1,000 IOC patterns, planted as bench.py plants them (seed 4321, 1,000 ppm);
 - configs[1]: the 32 dense patterns;
 - configs[4]: the 10,000 caseless patterns over long JSON-ish lines (an 8 MiB generated sample tiled to --c4-gib GiB);
 - -F IOC lists of 1k, 10k and 100k literals (tools/literal_probe.py) over 256 MiB of configs[1] text in which one line in
   2,000 gets " ioc=<literal>", repeated to --gib GiB.
Per set three runs, alternated over --rounds rounds after one warm-up round:
 1. `floor`: the count-only scan of the set (NULL callback; -F: gpugrep_literal_scan_buffer);
 2. `counts`: gpugrep_pattern_counts_buffer;
 3. `records`: today's route, gpugrep_scan_buffer with ids = index and flags | SINGLEMATCH (-F: the report scan with ids =
    index) and a callback that counts the records per id with numpy.  When one such call takes longer than --slow-s, that
    route runs in --slow-rounds rounds only (the entry says so).
Each reports the median and range of `gpu_ms` (device events around each segment's kernels, summed), the median host wall
time, launches and path; the compile times are the first calls of the floor and of the counts route on 4 KiB.  The counts
of routes 2 and 3 are compared.  The card's name and power limit are read in the same run.
Usage:
    python tools/pattern_counts_probe.py [--gib 2] [--c4-gib 1] [--sizes 1000,10000,100000] [--out profiles/pattern_counts_probe.json]
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gpu_api import Stats  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402
from literal_probe import iocs  # noqa: E402
from oracle_api import CALLBACK  # noqa: E402

_RECORD = np.dtype([("id", np.uint32), ("pad", np.uint32), ("line_number", np.uint64), ("line", np.uint64)])


def main() -> None:  # pylint: disable=too-many-locals,too-many-statements
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=2.0)
    ap.add_argument("--c4-gib", type=float, default=1.0)
    ap.add_argument("--sizes", default="1000,10000,100000")
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--slow-s", type=float, default=15.0)
    ap.add_argument("--slow-rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pattern_counts_probe.json"))
    args = ap.parse_args()
    import torch  # pylint: disable=import-outside-toplevel

    lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
    vp, u, i, ull = ctypes.c_void_p, ctypes.c_uint, ctypes.c_int, ctypes.c_ulonglong
    reg = lib.gpugrep_scan_buffer
    reg.restype, reg.argtypes = i, [vp, ctypes.c_size_t, i, vp, vp, vp, u, vp, i, i, ull, vp, vp]
    lit = lib.gpugrep_literal_scan_buffer
    lit.restype, lit.argtypes = i, [vp, ctypes.c_size_t, i, vp, vp, u, vp, i, i, ull, u, u, i, vp, vp]
    rep = lib.gpugrep_literal_report_scan_buffer
    rep.restype, rep.argtypes = i, [vp, ctypes.c_size_t, i, vp, vp, vp, u, vp, i, i, ull, vp, vp]
    cnt = lib.gpugrep_pattern_counts_buffer
    cnt.restype, cnt.argtypes = i, [vp, ctypes.c_size_t, i, vp, vp, u, i, i, vp, vp, vp]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=False).stdout.strip().splitlines()
    results = {"card": smi[0] if smi else "unknown", "rounds": args.rounds, "sets": []}
    per_id: list = [None]

    def on_batch(results_ptr, count):
        recs = np.ctypeslib.as_array(ctypes.cast(results_ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(count * _RECORD.itemsize,))
        ids = recs.view(_RECORD)["id"]
        per_id[0] += np.bincount(ids, minlength=per_id[0].size)[: per_id[0].size]

    callback = CALLBACK(on_batch)
    cb = ctypes.cast(callback, ctypes.c_void_p)

    def run(route: str, dev, size: int, arrays, fixed: bool) -> dict:
        pa, fa, fa_sm, ids, zeros, n = arrays
        st = Stats()
        counts = (ctypes.c_ulonglong * n)()
        per_id[0] = np.zeros(n, dtype=np.int64)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if route == "floor":
            rc = lit(dev, size, 1, pa, fa, n, None, 262140, 4096, 0, 0, 0, 0, None, ctypes.byref(st)) if fixed else \
                reg(dev, size, 1, pa, fa_sm, zeros, n, None, 262140, 4096, 0, None, ctypes.byref(st))
        elif route == "counts":
            rc = cnt(dev, size, 1, pa, fa, n, int(fixed), 262140, None, counts, ctypes.byref(st))
        else:
            rc = rep(dev, size, 1, pa, fa_sm, ids, n, cb, 262140, 4096, 0, None, ctypes.byref(st)) if fixed else \
                reg(dev, size, 1, pa, fa_sm, ids, n, cb, 262140, 4096, 0, None, ctypes.byref(st))
        wall = time.perf_counter() - t0
        out = {"route": route, "rc": rc, "gpu_ms": round(st.gpu_ms, 3), "wall_s": round(wall, 4), "launches": st.launches,
               "matches": st.matches, "path": st.path}
        if route == "counts":
            out["counts"] = list(counts)
        if route == "records":
            out["counts"] = per_id[0].tolist()
        return out

    def summary(samples: list[dict]) -> dict:
        ms = sorted(r["gpu_ms"] for r in samples)
        walls = sorted(r["wall_s"] for r in samples)
        out = {k: v for k, v in samples[-1].items() if k != "counts"}
        out.update({"gpu_ms": ms[len(ms) // 2], "gpu_ms_min": ms[0], "gpu_ms_max": ms[-1], "wall_s": walls[len(walls) // 2],
                    "wall_s_min": walls[0], "rounds": len(samples)})
        return out

    def measure(name: str, dev, size: int, patterns: list[bytes], flags: list[int], fixed: bool) -> None:
        n = len(patterns)
        pa = (ctypes.c_char_p * n)(*patterns)
        arrays = (pa, (u * n)(*flags), (u * n)(*[f | 8 for f in flags]), (u * n)(*range(n)), (u * n)(*([0] * n)), n)
        entry = {"set": name, "patterns": n, "bytes": size, "fixed": fixed}
        for route in ("floor", "counts"):   # the first call of each compiles (and caches) its databases
            t0 = time.perf_counter()
            run(route, dev, 4096, arrays, fixed)
            entry[f"{route}_compile_s"] = round(time.perf_counter() - t0, 3)
        runs: dict = {"floor": [], "counts": [], "records": []}
        slow = False
        for round_no in range(args.rounds + 1):   # (round 0 warms up)
            for route in runs:
                if route == "records" and slow and round_no > args.slow_rounds:
                    continue
                r = run(route, dev, size, arrays, fixed)
                assert r["rc"] == 0, (name, route, r["rc"])
                if route == "records" and r["wall_s"] > args.slow_s:
                    slow = True
                if round_no:
                    runs[route].append(r)
        assert runs["counts"][-1]["counts"] == runs["records"][-1]["counts"], name
        counts = runs["counts"][-1]["counts"]
        entry["patterns_seen"] = sum(1 for c in counts if c)
        entry["counted_lines"] = sum(counts)
        entry["runs"] = [summary(r) for r in runs.values()]
        entry["records_route_rounds_capped"] = slow
        floor = entry["runs"][0]["gpu_ms"]
        entry["counts_over_floor_gpu"] = round(entry["runs"][1]["gpu_ms"] / floor, 3) if floor else None
        entry["records_over_counts_wall"] = round(entry["runs"][2]["wall_s"] / entry["runs"][1]["wall_s"], 2)
        print(json.dumps(entry), flush=True)
        results["sets"].append(entry)

    size = int(args.gib * (1 << 30))
    c3, plants = synth.c3_patterns()
    host = torch.empty(size, dtype=torch.uint8)
    synth.fill_syslog(host.numpy(), seed=4321, plants=plants, plant_ppm=1000)
    host[-1] = 10
    dev = host.cuda()
    measure("configs[2] 1,000 IOC patterns, planted", dev.data_ptr(), size, [p.encode() for p in c3], [14] * len(c3), False)
    del dev
    synth.fill_syslog(host.numpy(), seed=1234)
    host[-1] = 10
    dev = host.cuda()
    measure("configs[1] 32 dense patterns", dev.data_ptr(), size, [p.encode() for p in synth.C2_PATTERNS], [14] * 32, False)
    base = synth.syslog_bytes(256 << 20, seed=7)
    for count in [int(s) for s in args.sizes.split(",")]:
        lits = iocs(count, seed=count)
        lines = base.split(b"\n")
        for k in range(0, len(lines) - 1, 2000):
            lines[k] += b" ioc=" + lits[(k // 2000) % len(lits)]
        pdev = torch.frombuffer(bytearray(b"\n".join(lines) * max(1, size // len(base))), dtype=torch.uint8).cuda()
        del lines
        measure(f"-F {count:,} IOC literals", pdev.data_ptr(), pdev.numel(), lits, [0] * len(lits), True)
        del pdev
        torch.cuda.empty_cache()
    del dev, host
    torch.cuda.empty_cache()
    c5 = synth.c5_patterns(10000)
    sample = np.frombuffer(synth.jsonish_bytes(8 << 20, patterns_to_plant=["session_4242 failed", "code=E31337abcd"]), dtype=np.uint8)
    long_size = int(args.c4_gib * (1 << 30))
    tiled = torch.from_numpy(np.tile(sample, -(-long_size // sample.size))[:long_size].copy())
    tiled[-1] = 10
    tdev = tiled.cuda()
    measure("configs[4] 10,000 caseless patterns, long lines", tdev.data_ptr(), long_size, [p.encode() for p in c5], [15] * len(c5), False)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as handle:
        json.dump(results, handle, indent=1)


if __name__ == "__main__":
    main()
