"""Fixed strings (grep -F) against the escaped-regex route on IOC-shaped lists; writes profiles/literal_probe.json.

Seeded configs[1] syslog (>= 2 GiB, device-resident) with planted hits.  Lists of 1k, 10k, 100k and 1M literals (IPv4s,
MD5 / SHA-256 hex, domains).  Per list: host compile time and device GB/s of gpugrep_literal_scan_buffer, and - where the
regex compiler takes the re.escape-d list (1k, 10k, 50k) - the same for gpugrep_context_scan_buffer, alternating the two
routes.  GB/s = bytes / wall time of the call (the input is resident, the callback counts only).  Usage:
    python tools/literal_probe.py [--gib 2] [--sizes 1000,10000,100000,1000000] [--out profiles/literal_probe.json]
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from gpu_api import Stats, marshal  # noqa: E402
from hypergrep_b200 import synth, utils  # noqa: E402


def iocs(count: int, seed: int) -> list[bytes]:
    rng = np.random.default_rng(seed)
    hexd = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)
    letters = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
    out = []
    for k in range(count):
        kind = k % 4
        if kind == 0:
            out.append(".".join(str(v) for v in rng.integers(1, 255, size=4)).encode())
        elif kind == 1:
            out.append(hexd[rng.integers(0, 16, size=32)].tobytes())
        elif kind == 2:
            out.append(hexd[rng.integers(0, 16, size=64)].tobytes())
        else:
            out.append(rng.choice(letters, size=int(rng.integers(6, 16))).tobytes() + b".example.net")
    return list(dict.fromkeys(out))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=2.0)
    ap.add_argument("--sizes", default="1000,10000,100000,1000000")
    ap.add_argument("--regex-max", type=int, default=50000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "literal_probe.json"))
    args = ap.parse_args()
    import torch  # pylint: disable=import-outside-toplevel

    lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
    lit_entry = lib.gpugrep_literal_scan_buffer
    lit_entry.restype = ctypes.c_int
    lit_entry.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                          ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p,
                          ctypes.c_void_p]
    ctx_entry = lib.gpugrep_context_scan_buffer
    ctx_entry.restype = ctypes.c_int
    ctx_entry.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                          ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int,
                          ctypes.c_void_p, ctypes.c_void_p]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=False).stdout.strip().splitlines()
    base = synth.syslog_bytes(256 << 20, seed=7)
    reps = max(1, int(args.gib * (1 << 30) // len(base)))
    results = {"card": smi[0] if smi else "unknown", "bytes": len(base) * reps, "lists": []}
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
        entry_res = {"literals": n}
        t0 = time.perf_counter()   # the first call compiles (and caches) the database; 4 KiB of text take no time
        st = Stats()
        rc = lit_entry(dev.data_ptr(), 4096, 1, la, None, n, None, 262140, 16, 0, 0, 0, 0, None, ctypes.byref(st))
        entry_res["literal_compile_s"] = time.perf_counter() - t0
        pats = [re.escape(lit.decode()) for lit in lits] if n <= args.regex_max else None
        if pats:
            pa, fa, ia, pn = marshal(pats, [8] * n, [0] * n)
            t0 = time.perf_counter()
            rc2 = lib.check_patterns(pa, fa, ia, pn)
            entry_res["regex_compile_s"] = time.perf_counter() - t0
            entry_res["regex_compile_rc"] = rc2
        runs = {"literal": [], "regex": []}
        for _ in range(args.reps):
            for route in ("literal", "regex"):
                if route == "regex" and not pats:
                    continue
                st = Stats()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if route == "literal":
                    rc = lit_entry(dev.data_ptr(), len(data), 1, la, None, n, None, 262140, 16, 0, 0, 0, 0, None, ctypes.byref(st))
                else:
                    rc = ctx_entry(dev.data_ptr(), len(data), 1, pa, fa, ia, pn, None, 262140, 16, 0, 0, 0, 0, None, ctypes.byref(st))
                wall = time.perf_counter() - t0
                runs[route].append({"rc": rc, "wall_s": wall, "gbps": len(data) / wall / 1e9, "matches": st.matches,
                                    "candidates_per_gib": st.candidates / (len(data) / (1 << 30)), "path": st.path, "launches": st.launches})
        entry_res.update(runs)
        if runs["regex"]:
            entry_res["same_count"] = all(a["matches"] == runs["regex"][0]["matches"] for a in runs["literal"] + runs["regex"])
        print(json.dumps(entry_res), flush=True)
        results["lists"].append(entry_res)
        del dev
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as handle:
        json.dump(results, handle, indent=1)


if __name__ == "__main__":
    main()
