"""Match events of the general path on the GPU (k_match_pl_events -> Job::deliver_events), and databases of many DFA groups.

a. Random general-mode cases (event_cases.event_case): records, return code and batch sizes == the oracle's, from a file,
   pageable, pinned and device memory, and in many segments.
b. Exact match ends: gpugrep_match_ends == oracle_ends_buffer, from host and device memory, across segments, and with a
   capacity below the count.
c. Sets of 31, 32, 33, 64 and 65 DFA groups plus NFA fallbacks: the 32-bit group mask of the fast path wraps past group 31,
   and group 31 shares bit 31 with the NFA patterns.  Then general mode over more than 32 groups.
d. The bound on the match events of one segment: a device-resident text of 200 MiB with a pattern that reports every
   letter is cut into pieces under the bound; a 64 MiB text denser than the bound still fails with 7.
"""

from __future__ import annotations

import ctypes
import functools

import numpy as np
import pytest

import event_cases as ec
import fast_path_cases as fpc
from gpu_api import Stats
from oracle_api import CALLBACK, load_oracle, run_scan, scan_bytes
from test_invert_match import compare_invert

pytestmark = pytest.mark.gpu

HOST, DEVICE = 0, 1
N_EVENT_CASES = 15


@pytest.fixture(scope="module")
def torch():
    import torch as module  # pylint: disable=import-outside-toplevel

    assert module.cuda.is_available()
    return module


@functools.lru_cache(maxsize=4)
def _case(seed: int) -> dict:
    return ec.event_case(seed, load_oracle())


def buffer_scan(lib, ptr: int, size: int, location: int, patterns, flags, ids, buffer_size=262140, buffer_count=16, max_match_count=0,
                collect=True, callback=None):
    """gpugrep_scan_buffer -> (rc, records, batch sizes, stats).  collect False: NULL callback (count-only); `callback`: a
    native callback address instead."""
    pa, fa, ia, n = ec._marshal(patterns, flags, ids)  # pylint: disable=protected-access
    lib.gpugrep_scan_buffer.restype = ctypes.c_int
    lib.gpugrep_scan_buffer.argtypes = [
        ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p,
    ]
    got, batches = [], []

    def cb(results, count):
        batches.append(count)
        for i in range(count):
            got.append((results[i].id, results[i].line_number, results[i].line))

    ccb = CALLBACK(cb) if collect and callback is None else None
    cb_ptr = callback if callback is not None else (ctypes.cast(ccb, ctypes.c_void_p) if ccb else None)
    stats = Stats()
    rc = lib.gpugrep_scan_buffer(ptr, size, location, pa, fa, ia, n, cb_ptr, buffer_size, buffer_count, max_match_count, None,
                                 ctypes.byref(stats))
    return rc, got, batches, stats


def _same(got, expected, label: str) -> None:
    if got != expected:
        for k, (a, b) in enumerate(zip(got, expected)):
            assert a == b, f"{label}: record {k}: got {a} expected {b}"
        raise AssertionError(f"{label}: {len(got)} records, the oracle has {len(expected)}")


def _inputs(torch, data: bytes):
    host = np.frombuffer(data, dtype=np.uint8)
    pinned = torch.from_numpy(host.copy()).pin_memory()
    dev = pinned.cuda()
    torch.cuda.synchronize()
    return host, pinned, dev


# ---- a. random general-mode cases ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(N_EVENT_CASES))
def test_random_event_cases_match_the_oracle(seed, gpu_lib, oracle_lib, torch, tmp_path, monkeypatch):
    """Records (ids, line numbers, texts, order), return code and batch sizes of a random general-mode case == the
    oracle's, from a file, pageable, pinned and device memory, and cut into many segments from a file and the device."""
    case = _case(seed)
    data, pats, flags, ids, bs, bc = case["data"], case["patterns"], case["flags"], case["ids"], case["buffer_size"], case["buffer_count"]
    path = tmp_path / "case.log"
    path.write_bytes(data)
    limit = case["max_match"]
    if limit == "mid":
        rc, full, _ = run_scan(oracle_lib, str(path), pats, flags, ids, buffer_size=bs, buffer_count=bc)
        assert rc == 0
        limit = ec.mid_line_limit(full)
    kw = {"buffer_size": bs, "buffer_count": bc, "max_match_count": limit}
    exp_rc, expected, exp_batches = run_scan(oracle_lib, str(path), pats, flags, ids, **kw)
    assert exp_rc == 0
    label = f"seed {seed} {pats} flags={flags} ids={ids} bs={bs} bc={bc} max={limit}"
    rc, got, batches = run_scan(gpu_lib, str(path), pats, flags, ids, **kw)
    assert rc == 0, label
    _same(got, expected, f"{label} file")
    assert batches == exp_batches, label
    host, pinned, dev = _inputs(torch, data)
    for what, ptr, loc in (("host", host.ctypes.data, HOST), ("pinned", pinned.data_ptr(), HOST), ("device", dev.data_ptr(), DEVICE)):
        rc, got, batches, st = buffer_scan(gpu_lib, ptr, len(data), loc, pats, flags, ids, **kw)
        assert rc == 0, f"{label} {what}"
        _same(got, expected, f"{label} {what}")
        assert batches == exp_batches, f"{label} {what}"
        assert st.path & 2, f"{label} {what}: path {st.path}"
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", str(max(1, len(data) // 7)))
    rc, got, batches = run_scan(gpu_lib, str(path), pats, flags, ids, **kw)
    assert rc == 0
    _same(got, expected, f"{label} file in segments")
    assert batches == exp_batches
    rc, got, batches, st = buffer_scan(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids, **kw)
    assert rc == 0
    _same(got, expected, f"{label} device in segments")
    assert batches == exp_batches
    assert st.segments > 1 or limit, f"{label}: {st.segments} segments"


# ---- b. exact match ends ------------------------------------------------------------------------------------------------

def _check_ends(gpu_lib, oracle_lib, data: bytes, dev, pats, flags, ids, bs: int, label: str, monkeypatch) -> int:
    """gpugrep_match_ends == oracle_ends_buffer from host and device memory, whole and in segments; a capacity below the
    count stores the first records and still returns the full count.  Returns the number of ends."""
    rc, expected, count = ec.oracle_ends(oracle_lib, data, pats, flags, ids, bs)
    assert rc == 0 and count == len(expected), label
    host = np.frombuffer(data, dtype=np.uint8)
    for chunk in ("", str(max(1, len(data) // 5))):
        monkeypatch.setenv("GPUGREP_CHUNK_BYTES", chunk)
        for what, ptr, loc in (("host", host.ctypes.data, HOST), ("device", dev.data_ptr(), DEVICE)):
            st = Stats()
            rc, got, found = ec.match_ends(gpu_lib, ptr, len(data), loc, pats, flags, ids, bs, capacity=count + 3, stats=st)
            assert rc == 0, f"{label} {what} {chunk}"
            _same(got, expected, f"{label} ends {what} chunk={chunk or 'default'}")
            assert found == count and st.matches == count
            assert st.path & 2 or count == 0
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "")
    if count > 1:
        cap = count // 2
        rc, got, found = ec.match_ends(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids, bs, capacity=cap)
        assert rc == 0 and found == count and got == expected[:cap], f"{label}: capacity {cap}"
    return count


@pytest.mark.parametrize("seed", range(N_EVENT_CASES))
def test_random_match_ends_match_the_oracle(seed, gpu_lib, oracle_lib, torch, monkeypatch):
    """Every (line, id, end) of a random case's set - variable width, anchors, caseless, NFA fallbacks, byte-alphabet
    patterns - equals the oracle's, SINGLEMATCH cleared."""
    case = _case(seed)
    _, _, dev = _inputs(torch, case["data"])
    _check_ends(gpu_lib, oracle_lib, case["data"], dev, case["patterns"], case["flags"], case["ids"], case["buffer_size"],
                f"seed {seed} {case['patterns']}", monkeypatch)


def test_match_ends_at_the_end_of_data(gpu_lib, oracle_lib, torch, monkeypatch):
    """Ends that the DFA reports on the end-of-data transition ($, \\b, \\z at the end of a block, after a NUL, at the end
    of a pseudo-line cut by buffer_size, at the end of a text without a final newline), and variable-width patterns."""
    pats = [r"ab$", r"b\b", r"[ab]+\z", r"(?i)B\Z", r"a+", r"x*y", r"\w{2,3}$"]
    flags = [0, 4, 0, 0, 0, 0, 2]
    ids = [1, 2, 3, 4, 5, 6, 7]
    data = b"ab\nab ab\nb\0ab\nzzab ab\nxxy abab\n" * 4000 + b"aaabbb aab" * 300 + b"\nab"
    _, _, dev = _inputs(torch, data)
    for bs in (262140, 64, 9):
        assert _check_ends(gpu_lib, oracle_lib, data, dev, pats, flags, ids, bs, f"end-of-data bs={bs}", monkeypatch) > 10000


# ---- c. many DFA groups -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("k", [31, 32, 33, 64, 65])
def test_many_groups_fast_path(k, gpu_lib, oracle_lib, torch, tmp_path):
    """k one-word DFA groups plus two NFA fallbacks in simple mode: the members of groups 0, 31, 32, 63, 64 and k - 1 and the NFA
    patterns, planted at every offset mod 16, are found by default (fast path, local walk with the NFA and k_confirm), with
    GPUGREP_FORCE_GENERAL, with GPUGREP_NFA_GENERAL, inverted and count-only - each time the oracle's records."""
    groups = ec.many_group_set(gpu_lib, k, "simple")
    assert groups["groups"] == k and groups["simple"] and groups["nfa"] == 2
    pats, flags, ids = groups["patterns"], groups["flags"], groups["ids"]
    data = ec.many_group_text(groups, seed=k)
    budget = {"GPUGREP_MAX_DFA_STATES": str(groups["budget"])}
    with fpc.environment(budget):
        rc, expected, _ = scan_bytes(oracle_lib, data, pats, flags=flags, ids=ids)
        assert rc == 0
        lines = [text for _, _, text in expected]
        for g, word in groups["member"].items():
            alone = [t for t in lines if word.encode() in t and b"kilo" not in t]
            assert len(alone) >= 16, f"group {g}: {len(alone)} lines"
        assert sum(1 for t in lines if b"omega" in t) >= 16 and sum(1 for t in lines if b"gram" in t) >= 32
        pred = fpc.predict(gpu_lib, pats, flags, ids, budget, data, 262140)
        assert pred["groups"] == k and pred["nfa"] == 2 and pred["fast"]
        assert pred["verify"] == "local_nfa+confirm", pred.get("verify")
        host, _, dev = _inputs(torch, data)
        for what, ptr, loc in (("host", host.ctypes.data, HOST), ("device", dev.data_ptr(), DEVICE)):
            rc, got, _, st = buffer_scan(gpu_lib, ptr, len(data), loc, pats, flags, ids)
            assert rc == 0
            _same(got, expected, f"k={k} {what}")
            assert st.path == pred["path"] == 1, st.path
            if what == "device":
                assert st.segments == 1 and st.launches == 9 + pred["confirm"], st.launches
        for switch in ("GPUGREP_FORCE_GENERAL", "GPUGREP_NFA_GENERAL"):
            with fpc.environment({switch: "1"}):
                rc, got, _, st = buffer_scan(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids)
            assert rc == 0
            _same(got, expected, f"k={k} {switch}")
            assert st.path == 2, (switch, st.path)
        rc, _, _, st = buffer_scan(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids, collect=False)
        assert rc == 0 and st.matches == len(expected) and st.path == 1
        compare_invert(gpu_lib, oracle_lib, data, pats, flags, ids, tmp_dir=str(tmp_path))


@pytest.mark.parametrize("k", [32, 33, 65])
def test_many_groups_general_mode(k, gpu_lib, oracle_lib, torch, tmp_path, monkeypatch):
    """k one-word groups with distinct ids, every other word without SINGLEMATCH, plus NFA fallbacks: the reports of every
    group are flattened (accept_base) and expanded to ids on the host - records and match ends == the oracle's."""
    groups = ec.many_group_set(gpu_lib, k, "general", extra_nfa=2)
    assert groups["groups"] == k and not groups["simple"] and groups["nfa"] == 4
    pats, flags, ids = groups["patterns"], groups["flags"], groups["ids"]
    data = ec.many_group_text(groups, seed=100 + k, size=512 << 10)
    path = tmp_path / "groups.log"
    path.write_bytes(data)
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", str(groups["budget"]))
    rc, expected, exp_batches = run_scan(oracle_lib, str(path), pats, flags, ids)
    assert rc == 0 and len({i for i, _, _ in expected}) == len(groups["member"]) + 4
    rc, got, batches = run_scan(gpu_lib, str(path), pats, flags, ids)
    assert rc == 0
    _same(got, expected, f"k={k} general file")
    assert batches == exp_batches
    _, _, dev = _inputs(torch, data)
    rc, got, _, st = buffer_scan(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids)
    assert rc == 0 and st.path == 2
    _same(got, expected, f"k={k} general device")
    _check_ends(gpu_lib, oracle_lib, data, dev, pats, flags, ids, 262140, f"k={k} general ends", monkeypatch)


# ---- d. the event bound of one segment ----------------------------------------------------------------------------------

def test_dense_events_of_a_large_device_buffer(gpu_lib, torch):
    """200 MiB of lowercase lines on the device and `[a-z]` without SINGLEMATCH: about 2 * 10^8 events, more than one
    segment holds (2^27).  The 2 GiB device segment is scanned again in 64 MiB pieces: count-only, with a native callback
    and gpugrep_match_ends all count every letter, like a scan of the same bytes from host memory, and the first 2^20 ends
    are those of a numpy model."""
    n = 200 << 20
    gen = torch.Generator(device="cuda").manual_seed(20)
    text = torch.randint(97, 123, (n,), dtype=torch.uint8, device="cuda", generator=gen)
    text[torch.rand(n, device="cuda", generator=gen) < 1.0 / 48] = 10
    text[-1] = 10
    letters = int((text != 10).sum().item())
    assert letters > (1 << 27)
    torch.cuda.synchronize()
    pats, flags, ids = ["[a-z]"], [0], [1]
    rc, _, _, st = buffer_scan(gpu_lib, text.data_ptr(), n, DEVICE, pats, flags, ids, collect=False)
    assert rc == 0, gpu_lib.gpugrep_last_error()
    assert st.matches == letters and st.split_segments == 1 and st.path == 2
    discard = ctypes.cast(gpu_lib.gpugrep_discard_results, ctypes.c_void_p).value
    rc, _, _, st = buffer_scan(gpu_lib, text.data_ptr(), n, DEVICE, pats, flags, ids, callback=discard, buffer_count=4096)
    assert rc == 0 and st.matches == letters and st.split_segments == 1
    host = text.cpu().numpy()
    rc, _, _, st = buffer_scan(gpu_lib, host.ctypes.data, n, HOST, pats, flags, ids, collect=False)
    assert rc == 0 and st.matches == letters and st.split_segments == 0
    entry = ec.ends_entry(gpu_lib)
    pa, fa, ia, cnt = ec._marshal(pats, flags, ids)  # pylint: disable=protected-access
    found = ctypes.c_size_t()
    assert entry(text.data_ptr(), n, DEVICE, pa, fa, ia, cnt, 262140, None, 0, ctypes.byref(found), None) == 0
    assert found.value == letters
    cap = 1 << 20
    out = np.zeros(cap, dtype=[("line", "<u8"), ("id", "<u4"), ("end", "<u4")])
    assert entry(text.data_ptr(), n, DEVICE, pa, fa, ia, cnt, 262140, out.ctypes.data, cap, ctypes.byref(found), None) == 0
    assert found.value == letters
    head = host[: 4 << 20]
    pos = np.flatnonzero(head != 10)[:cap]
    newlines = np.flatnonzero(head == 10)
    line = np.searchsorted(newlines, pos)
    start = np.where(line > 0, newlines[np.maximum(line, 1) - 1] + 1, 0)
    assert pos.size == cap
    assert np.array_equal(out["line"], line) and np.array_equal(out["end"], pos - start + 1) and np.all(out["id"] == 1)


def test_events_denser_than_the_bound_fail_with_7(gpu_lib, monkeypatch):
    """The bound that remains: a 64 MiB piece with three patterns that each report every letter, in three DFA groups, has
    about 2 * 10^8 events - more than 2^27.  The scan fails with 7 and says why."""
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", "6")
    pats, flags, ids = ["[a-z]", "[b-y]", "[c-x]"], [0, 0, 0], [1, 2, 3]
    from dfa_sim import CompiledDb  # pylint: disable=import-outside-toplevel

    assert CompiledDb(gpu_lib, pats, flags, ids).info.groups == 3
    rng = np.random.default_rng(64)
    host = rng.integers(97, 123, 64 << 20, dtype=np.uint8)
    host[rng.random(host.size) < 1.0 / 64] = 10
    host[-1] = 10
    rc, _, _, _ = buffer_scan(gpu_lib, host.ctypes.data, host.size, HOST, pats, flags, ids, collect=False)
    gpu_lib.gpugrep_last_error.restype = ctypes.c_char_p
    assert rc == 7 and b"too many match events" in gpu_lib.gpugrep_last_error()
