"""Run as a subprocess by tests/test_gpu_parity.py::test_device_text_reads_stay_inside_the_buffer.

compute-sanitizer is not available on the GPU pool, so the bound on caller-owned device text is checked with the
hardware: the text is placed in a virtual-memory mapping (cuMemAddressReserve / cuMemMap) whose neighbouring pages are
reserved but NOT mapped, flush against the end (and then the start) of the mapping.  A kernel that reads one byte past
data + round_up(size, 16) - the contract of GPUGREP_LOC_DEVICE in include/gpugrep.h - or before `data` takes an illegal
address fault, the scan returns 7 and this process exits non-zero.  Results are compared with the oracle as well.
"""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
from cuda.bindings import driver  # noqa: E402

from gpu_api import scan_buffer  # noqa: E402
from hypergrep_b200 import synth  # noqa: E402
from oracle_api import load_oracle, scan_bytes  # noqa: E402


def ok(result):
    code, *rest = result
    assert code == driver.CUresult.CUDA_SUCCESS, code
    return rest[0] if len(rest) == 1 else rest


def main() -> int:
    torch.zeros(1, device="cuda:0")   # primary context
    lib = ctypes.CDLL(os.path.join(ROOT, "hypergrep_b200", "lib", "libgpugrep.so"))
    lib.gpugrep_last_error.restype = ctypes.c_char_p
    oracle = load_oracle()
    prop = driver.CUmemAllocationProp()
    prop.type = driver.CUmemAllocationType.CU_MEM_ALLOCATION_TYPE_PINNED
    prop.location.type = driver.CUmemLocationType.CU_MEM_LOCATION_TYPE_DEVICE
    prop.location.id = 0
    gran = ok(driver.cuMemGetAllocationGranularity(prop, driver.CUmemAllocationGranularity_flags.CU_MEM_ALLOC_GRANULARITY_MINIMUM))
    pages = 8   # 16 MiB with the usual 2 MiB granularity
    base = int(ok(driver.cuMemAddressReserve((pages + 2) * gran, 0, 0, 0)))
    handle = ok(driver.cuMemCreate(pages * gran, prop, 0))
    lo, hi = base + gran, base + gran + pages * gran
    ok(driver.cuMemMap(lo, pages * gran, 0, handle, 0))
    access = driver.CUmemAccessDesc()
    access.location.type = driver.CUmemLocationType.CU_MEM_LOCATION_TYPE_DEVICE
    access.location.id = 0
    access.flags = driver.CUmemAccess_flags.CU_MEM_ACCESS_FLAGS_PROT_READWRITE
    ok(driver.cuMemSetAccess(lo, pages * gran, [access], 1))
    # the neighbours really are unmapped: a copy out of them is refused
    probe = (ctypes.c_char * 16)()
    assert driver.cuMemcpyDtoH(probe, hi, 16)[0] != driver.CUresult.CUDA_SUCCESS
    assert driver.cuMemcpyDtoH(probe, lo - 16, 16)[0] != driver.CUresult.CUDA_SUCCESS

    syslog = synth.syslog_bytes(6 << 20, seed=41)
    long_lines = synth.jsonish_bytes(3 << 20, patterns_to_plant=["session_4242 failed"])
    c3, plants = synth.c3_patterns()
    planted = synth.syslog_bytes(4 << 20, seed=43, plants=plants, plant_ppm=2000)
    c5 = synth.c5_patterns(600)
    cases = [
        ("C2 fast path", syslog, synth.C2_PATTERNS, None, None),
        ("C1 stride 4", syslog, synth.C1_PATTERNS, None, None),
        ("C3 confirm + groups", planted, c3, None, None),
        ("C5 caseless, long lines", long_lines, c5, [15] * len(c5), None),
        ("general path (ids, no singlematch)", syslog[: 2 << 20], ["ERROR", "port [0-9]+", "user=\\w+"], [6, 14, 6], [1, 2, 3]),
        ("NFA pattern on the fast path", syslog[: 3 << 20], ["Failed password", "user=.{40,60}port"], None, None),
        ("no newline at the end", syslog[: (1 << 20) + 5].rstrip(b"\n") + b" ERROR tail", synth.C2_PATTERNS, None, None),
        ("tiny", b"ERROR\n", synth.C1_PATTERNS, None, None),
    ]
    checked = 0
    for name, text, patterns, flags, ids in cases:
        for cut in ((0, 7) if len(patterns) > 100 else (0, 1, 7, 15)):   # sizes that are / are not multiples of 16
            data = text[: len(text) - cut] if cut else text
            n = len(data)
            padded = (n + 15) & ~15
            expected = scan_bytes(oracle, data, patterns, flags=flags, ids=ids)
            for where, ptr in (("end", hi - padded), ("start", lo)):
                ok(driver.cuMemsetD8(lo, 0x41, pages * gran))
                ok(driver.cuMemcpyHtoD(ptr, data, n))
                rc, got, stats = scan_buffer(lib, ptr, n, 1, patterns, flags=flags, ids=ids)
                if rc != 0:
                    print(f"FAIL {name} cut={cut} at {where}: rc={rc} {lib.gpugrep_last_error()}")
                    return 1
                if (rc, got) != (expected[0], expected[1]):
                    print(f"FAIL {name} cut={cut} at {where}: {len(got)} records, oracle {len(expected[1])}")
                    return 1
                checked += 1
    torch.cuda.synchronize()
    print(f"guarded scans ok: {checked}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
