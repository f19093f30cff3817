#!/usr/bin/env python3
"""One-off stress run: random parity cases (tests/parity.py) for a range of seeds against the oracle, on the GPU box.

    fuzz_gpu.py FIRST LAST          small random cases (parity.random_case)
    fuzz_gpu.py FIRST LAST text     benchmark pattern sets over synthetic text
    fuzz_gpu.py FIRST LAST bytes    the byte-alphabet cases (tests/byte_cases.py): random cases on both paths and on the
                                    NFA, and every 25th seed a factor set on the fast path
"""
import ctypes
import os
import sys
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import parity  # noqa: E402
from hypergrep_b200 import utils  # noqa: E402
from oracle_api import load_oracle  # noqa: E402

first, last = int(sys.argv[1]), int(sys.argv[2])
gpu = utils._get_hyperscanner_lib()
oracle = load_oracle()
bad = skipped = 0
for seed in (range(first, last) if len(sys.argv) <= 3 else ()):
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        skipped += 1
        continue
    try:
        parity.compare(gpu, oracle, data, patterns, flags, ids, buffer_size, buffer_count, max_match)
    except Exception:  # pylint: disable=broad-except
        bad += 1
        print(f"seed {seed} FAILED: patterns={patterns!r} flags={flags} ids={ids} buffer_size={buffer_size}")
        traceback.print_exc(limit=2)
        if bad >= 5:
            break
print(f"seeds {first}..{last}: {bad} failures, {skipped} skipped")


def text_mode(first: int, last: int) -> None:
    """Random subsets of the benchmark pattern sets over 0.5-3 MiB of synthetic syslog / JSON-ish text, random
    buffer sizes and segment sizes: exercises segment cuts, dense candidate lists, several DFA groups, long lines."""
    import random

    from hypergrep_b200 import synth

    c3, plants = synth.c3_patterns()
    c5 = synth.c5_patterns(400)
    pool = synth.C2_PATTERNS + synth.C1_PATTERNS + c3[:300] + c5[:200] + [r"\d{3,5} in lib\w+", r"(?i)failed \w+ for", r"^\w{3} +\d+ ", r"ssh2$"]
    failures = 0
    for seed in range(first, last):
        rng = random.Random(seed)
        k = rng.choice([1, 1, 2, 3, 8, 32, 120])
        patterns = rng.sample(pool, k)
        flags = [rng.choice([14, 14, 15])] * k
        size = rng.choice([1 << 19, 1 << 20, 3 << 20])
        if rng.random() < 0.3:
            data = synth.jsonish_bytes(size // 2, seed=seed, patterns_to_plant=["session_4242 failed", "code=E31337abcd"], plant_rate=0.3)
        else:
            data = synth.syslog_bytes(size, seed=seed, plants=plants[:50] if rng.random() < 0.5 else None, plant_ppm=20000, lib=gpu)
        os.environ["GPUGREP_CHUNK_BYTES"] = str(rng.choice([1, 1, 300000, 1 << 20]))   # test hook: tiny segments
        buffer_size = rng.choice([262140, 262140, 4096, 300, 64])
        try:
            parity.compare(gpu, oracle, data, patterns, flags=flags, buffer_size=buffer_size, buffer_count=rng.choice([16, 7, 1000]),
                           max_match_count=rng.choice([0, 0, 5, 1000]))
        except Exception:  # pylint: disable=broad-except
            failures += 1
            print(f"text seed {seed} FAILED: k={k} buffer_size={buffer_size} chunk={os.environ['GPUGREP_CHUNK_BYTES']} patterns={patterns[:4]!r}...")
            traceback.print_exc(limit=2)
            if failures >= 5:
                break
    print(f"text seeds {first}..{last}: {failures} failures")


if len(sys.argv) > 3 and sys.argv[3] == "text":
    text_mode(first, last)


def bytes_mode(first: int, last: int) -> None:
    """byte_random_case on the default path, with GPUGREP_FORCE_GENERAL=1 and with GPUGREP_MAX_DFA_STATES=3; every 25th seed
    also byte_fast_case (records of a file scan and of device input, count-only)."""
    import numpy as np

    import byte_cases
    import fast_path_cases as fpc
    from gpu_api import scan_buffer
    from oracle_api import scan_bytes

    failures = cases = 0
    for seed in range(first, last):
        patterns, flags, ids, buffer_size, data, buffer_count, max_match = byte_cases.byte_random_case(seed)
        if parity.has_all_nul_pseudo_line(data, buffer_size):
            continue
        for env in ({}, {"GPUGREP_FORCE_GENERAL": "1"}, {"GPUGREP_MAX_DFA_STATES": "3"}):
            cases += 1
            try:
                with fpc.environment(env):
                    parity.compare(gpu, oracle, data, patterns, flags, ids, buffer_size, buffer_count, max_match)
            except Exception:  # pylint: disable=broad-except
                failures += 1
                print(f"bytes seed {seed} {env} FAILED: patterns={patterns!r} flags={flags} ids={ids} buffer_size={buffer_size}")
                traceback.print_exc(limit=2)
        if seed % 25 == 0:
            case = byte_cases.byte_fast_case(seed)
            cases += 1
            try:
                rc, expected, _ = scan_bytes(oracle, case["data"], case["patterns"], flags=case["flags"], ids=case["ids"], buffer_size=case["buffer_size"])
                assert rc == 0
                parity.compare(gpu, oracle, case["data"], case["patterns"], case["flags"], case["ids"], case["buffer_size"])
                import torch

                dev = torch.from_numpy(np.frombuffer(case["data"], dtype=np.uint8).copy()).cuda()
                torch.cuda.synchronize()
                rc, got, _ = scan_buffer(gpu, dev.data_ptr(), len(case["data"]), 1, case["patterns"], case["flags"], case["ids"], buffer_size=case["buffer_size"])
                assert rc == 0 and got == expected
                rc, _, st = scan_buffer(gpu, dev.data_ptr(), len(case["data"]), 1, case["patterns"], case["flags"], case["ids"], collect=False,
                                        buffer_size=case["buffer_size"])
                assert rc == 0 and st.matches == len(expected)
            except Exception:  # pylint: disable=broad-except
                failures += 1
                print(f"bytes fast seed {seed} FAILED: patterns={case['patterns'][:4]!r}")
                traceback.print_exc(limit=2)
        if failures >= 5:
            break
    print(f"bytes seeds {first}..{last}: {cases} cases, {failures} failures")


if len(sys.argv) > 3 and sys.argv[3] == "bytes":
    bytes_mode(first, last)
