"""CPU side of the match-event tests (tests/test_match_events_gpu.py): the oracle's match ends against its own scans, the
random general-mode cases and their match ends through the host logic (Job::deliver_events) over the CPU engine mock, and
the group counts of the many-group sets."""

from __future__ import annotations

import collections

import numpy as np
import pytest

import event_cases as ec
import parity
from oracle_api import scan_bytes

CPU_SEEDS = range(12)
CPU_SIZE = 96 << 10


@pytest.mark.parametrize("seed", CPU_SEEDS)
def test_oracle_ends_agree_with_its_scan(seed, oracle_lib):
    """For an id without SINGLEMATCH, hyperscan() delivers one record per match end: oracle_ends_buffer's count per
    (line, id) equals hyperscan()'s record count per (line, id); every id with SINGLEMATCH has a record exactly on the
    lines where it has an end."""
    case = ec.event_case(seed, oracle_lib, size=CPU_SIZE)
    pats, flags, ids, bs = case["patterns"], case["flags"], case["ids"], case["buffer_size"]
    rc, records, _ = scan_bytes(oracle_lib, case["data"], pats, flags=flags, ids=ids, buffer_size=bs)
    assert rc == 0
    rc, ends, count = ec.oracle_ends(oracle_lib, case["data"], pats, flags, ids, bs)
    assert rc == 0 and count == len(ends)
    assert ends == sorted(ends, key=lambda e: (e[0], e[2], e[1])) and len(set(ends)) == len(ends)
    singlematch = {i for i, f in zip(ids, flags) if f & ec.SINGLEMATCH}
    per_ends = collections.Counter((line, i) for line, i, _ in ends)
    per_records = collections.Counter((line, i) for i, line, _ in records)
    assert {key: n for key, n in per_ends.items() if key[1] not in singlematch} == \
        {key: n for key, n in per_records.items() if key[1] not in singlematch}
    assert {key for key in per_ends if key[1] in singlematch} == {key for key in per_records if key[1] in singlematch}
    assert all(per_records[key] == 1 for key in per_records if key[1] in singlematch)
    rc, first, total = ec.oracle_ends(oracle_lib, case["data"], pats, flags, ids, bs, capacity=count // 3)
    assert rc == 0 and total == count and first == ends[: count // 3]


@pytest.mark.parametrize("seed", CPU_SEEDS)
def test_random_event_cases_on_the_host_logic(seed, hostmock_lib, oracle_lib):
    """The host logic over the CPU engine mock: records, batches and return code of a random general-mode case == the
    oracle's, and its match ends == oracle_ends_buffer (all of them, and the first third with the full count)."""
    case = ec.event_case(seed, oracle_lib, size=CPU_SIZE)
    pats, flags, ids, bs = case["patterns"], case["flags"], case["ids"], case["buffer_size"]
    limit = case["max_match"]
    if limit == "mid":
        _, full, _ = scan_bytes(oracle_lib, case["data"], pats, flags=flags, ids=ids, buffer_size=bs)
        limit = ec.mid_line_limit(full)
    parity.compare(hostmock_lib, oracle_lib, case["data"], pats, flags=flags, ids=ids, buffer_size=bs,
                   buffer_count=case["buffer_count"], max_match_count=limit)
    rc, expected, count = ec.oracle_ends(oracle_lib, case["data"], pats, flags, ids, bs)
    assert rc == 0
    host = np.frombuffer(case["data"], dtype=np.uint8)
    for capacity in (None, count // 3):
        rc, got, found = ec.match_ends(hostmock_lib, host.ctypes.data, host.size, 0, pats, flags, ids, bs, capacity=capacity)
        assert rc == 0 and found == count
        assert got == expected[: len(got)] and len(got) == (count if capacity is None else capacity)


@pytest.mark.parametrize("mode", ["simple", "general"])
@pytest.mark.parametrize("k", [31, 32, 33, 64, 65])
def test_many_group_sets(k, mode, hostmock_lib, oracle_lib):
    """many_group_set compiles to exactly k DFA groups (one word each) plus its NFA fallbacks in both modes, and the text
    plants every group member it names and every NFA pattern at each offset mod 16."""
    groups = ec.many_group_set(hostmock_lib, k, mode)
    assert groups["groups"] == k and groups["nfa"] == 2 and groups["simple"] == (mode == "simple")
    assert sorted(groups["member"]) == sorted({g for g in (0, 31, 32, 63, 64, k - 1) if g < k})
    data = ec.many_group_text(groups, seed=k, size=256 << 10)
    for piece in [w.encode() for w in groups["member"].values()] + [b"omega", b"kilo"]:
        offsets = set()
        at = data.find(piece)
        while at >= 0:
            offsets.add(at % 16)
            at = data.find(piece, at + 1)
        assert offsets == set(range(16)), piece
