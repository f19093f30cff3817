#!/usr/bin/env python3
"""Benchmark of the scan hot path (BASELINE.json metric: scanned GB/s; configs[1] = 32 mixed patterns over 10 GiB).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--gib G] [--strong] [--no-extras]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the hot path over one batch of synthetic syslog text (per rank: --gib GiB, default 10).
  value      : device-resident whole-job throughput, CUDA events on the stream the kernels run on, max over ranks.
  e2e        : same pass through the C ABI from PINNED HOST memory, H2D of the input and D2H of the records inside the
               timed region, full delivery path (matched lines copied into result slots, native discard callback).
  e2e_file   : the reference-facing call itself, hyperscan(path)-equivalent on a tmpfs file.
  e2e_python : hypergrep_b200.grep(path, count_only=True) and hypergrep_b200.scan(path, python callback, buffer_count=16).
  roofline   : the streaming kernel (k_stream) against the measured HBM copy peak (MEASURED_PEAKS.json).
  parity     : the matched line numbers of the timed text (a bounded prefix) equal the oracle's, order included.
  --dump-outputs DIR: what the last timed step computed, for comparing two builds on the same seeded text (see
               dump_outputs).
  extra      : device-resident throughput of BASELINE configs[0], [2], [4] and the configs[3] file leg (N=1 only).
  cpu_baseline / --impl reference: the oracle port (reference loop shape, PCRE2-JIT matcher; the reference itself needs
               Hyperscan, which is not installable here) on the box's host cores, bounded sample.
Multi-GPU: ranks scan independent newline-aligned shards, no collective on the data path.  Default: weak scaling
(rank-specific text).  --strong: ONE text of --gib GiB, rank r scans byte range r of N, the line numbers are rebased
with a prefix sum of the shard line counts (the only exchange) and the merged sequence is checked against a single-GPU
pass of the whole text on rank 0.
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD = "configs[1]: 32 mixed literal + character-class patterns, synthetic syslog text"
BLOCK = 16 << 20   # corpus generation granularity (hypergrep_b200.synth): every block ends on a line end


def parse_args() -> argparse.Namespace:
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=5)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="ours", choices=["ours", "reference"])
    parser.add_argument("--gib", type=float, default=float(os.environ.get("GPUGREP_BENCH_GIB", "10")))
    parser.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the cpu_baseline sample")
    parser.add_argument("--strong", action="store_true", help="one text of --gib GiB split over the ranks, merged and checked")
    parser.add_argument("--no-extras", action="store_true", help="skip the extra configs / Python-level legs")
    parser.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    return parser.parse_args()


def load_peaks() -> tuple[float, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path, encoding="utf-8") as handle:
            return float(json.load(handle)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (100 ms period: eight ranks polling at 20 ms took
    measurable host time from the scan threads on a 32-vCPU box)."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int) -> None:
        self.device = device
        self.proc = None
        self.lines: list[tuple[float, str]] = []
        self.windows: list[tuple[float, float]] = []   # timed regions (perf_counter), samples outside them are dropped

    def wait_first(self, timeout: float = 10.0) -> None:
        """nvidia-smi takes a second or more to print its first sample; the timed regions are shorter than that."""
        deadline = time.perf_counter() + timeout
        while self.proc is not None and not self.lines and time.perf_counter() < deadline:
            time.sleep(0.02)

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(  # pylint: disable=consider-using-with
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._drain, daemon=True).start()
        except OSError:
            self.proc = None

    def _drain(self) -> None:
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [(when, line) for when, line in self.lines if any(lo <= when <= hi for lo, hi in self.windows)]
        for when, line in (inside or self.lines):   # regions shorter than the sampling period: fall back to all samples
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, flag in zip(names, parts[5:9]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_inside_timed_regions": len(inside)}


# ---------------------------------------------------------------------------------------------------------------------
# oracle helpers (CPU): used by the parity check, the cpu_baseline leg and the reference arm only
# ---------------------------------------------------------------------------------------------------------------------
def marshal(patterns, flags=None):
    n = len(patterns)
    pa = (ctypes.c_char_p * n)(*[p.encode() for p in patterns])
    fa = (ctypes.c_uint * n)(*(flags or [14] * n))
    ia = (ctypes.c_uint * n)(*([0] * n))
    return pa, fa, ia, n


def load_oracle() -> ctypes.CDLL:
    path = os.path.join(ROOT, "oracle", "_build", "liboracle_hyperscanner.so")
    if not os.path.exists(path):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    lib = ctypes.CDLL(path)
    lib.oracle_count_buffer.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.oracle_lines_buffer.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
    return lib


def shard_bounds(view, size: int, shards: int) -> list[int]:
    """Newline-aligned shard boundaries of a byte buffer (numpy uint8 view)."""
    bounds = [0]
    for t in range(1, shards):
        pos = size * t // shards
        while pos < size and view[pos - 1] != 10:
            pos += 1
        bounds.append(max(pos, bounds[-1]))
    bounds.append(size)
    return bounds


def oracle_scan(oracle, view, size: int, patterns, threads: int, want_lines: bool, flags=None):
    """Oracle port (reference loop + PCRE2-JIT) over `threads` newline-aligned shards of view[0:size], all at once.
    Returns (wall seconds, matches, line numbers as one numpy array in file order or None)."""
    import numpy as np  # pylint: disable=import-outside-toplevel

    pa, fa, ia, n = marshal(patterns, flags)
    bounds = shard_bounds(view, size, threads)
    base = view.ctypes.data
    matches = [0] * threads
    lines = [0] * threads
    found: list = [None] * threads

    def work(t: int) -> None:
        m, ln = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        lo, hi = bounds[t], bounds[t + 1]
        if want_lines:
            cap = (hi - lo) // 64 + 1024
            out = np.empty(cap, dtype=np.uint64)
            rc = oracle.oracle_lines_buffer(base + lo, hi - lo, pa, fa, ia, n, 262140, out.ctypes.data, cap, ctypes.byref(m), ctypes.byref(ln))
            assert rc == 0 and m.value <= cap
            found[t] = out[: m.value]
        else:
            rc = oracle.oracle_count_buffer(base + lo, hi - lo, pa, fa, ia, n, 262140, ctypes.byref(m), ctypes.byref(ln))
            assert rc == 0
        matches[t], lines[t] = m.value, ln.value

    t0 = time.perf_counter()
    pool = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for th in pool:
        th.start()
    for th in pool:
        th.join()
    elapsed = time.perf_counter() - t0
    merged = None
    if want_lines:
        parts, base_line = [], 0
        for t in range(threads):
            parts.append(found[t] + np.uint64(base_line))
            base_line += lines[t]
        merged = np.concatenate(parts) if parts else np.empty(0, dtype=np.uint64)
    return elapsed, sum(matches), merged


def oracle_throughput(oracle, view, size: int, patterns, threads: int, seconds: float):
    """(GB/s, sample bytes, matches, wall seconds): the sample grows until it costs about `seconds` of wall time."""
    sample = min(size, (8 << 20) * threads)
    while sample > 1 and view[sample - 1] != 10:
        sample -= 1
    elapsed, matches, _ = oracle_scan(oracle, view, sample, patterns, threads, False)
    if elapsed < seconds / 3 and sample < size:
        scaled = min(size, int(sample * seconds / max(elapsed, 1e-3)))
        while scaled > 1 and view[scaled - 1] != 10:
            scaled -= 1
        sample = scaled
        elapsed, matches, _ = oracle_scan(oracle, view, sample, patterns, threads, False)
    return sample / elapsed / 1e9, sample, matches, elapsed


# ---------------------------------------------------------------------------------------------------------------------
def reference_arm(args, config: dict, patterns) -> None:
    """The reference's CPU implementation of the path (oracle port: the reference loop with PCRE2-JIT standing in for
    Hyperscan) on all host cores.  Loads libgpugrep_synth.so for the corpus and the oracle - never the product library."""
    import numpy as np  # pylint: disable=import-outside-toplevel

    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    oracle = load_oracle()
    threads = os.cpu_count() or 1
    total = args.warmup + args.steps
    size = int(args.gib * (1 << 30))
    text = np.empty(size, dtype=np.uint8)
    synth.fill_syslog(text, seed=1234)
    # the whole configured text per step if that fits the time budget (about two minutes for all steps), else a prefix
    probe_s, _, _ = oracle_scan(oracle, text, min(size, (16 << 20) * threads), patterns, threads, False)
    rate = min(size, (16 << 20) * threads) / max(probe_s, 1e-3)
    budget = max(2.0, 120.0 / max(1, total))
    sample = size if size / rate <= budget else int(rate * budget)
    while sample > 1 and text[sample - 1] != 10:
        sample -= 1
    rates, matches = [], 0
    for step in range(total):
        elapsed, matches, _ = oracle_scan(oracle, text, sample, patterns, threads, False)
        if step >= args.warmup:
            rates.append(sample / elapsed / 1e9)
    value = sum(rates) / len(rates)
    line = {
        "impl": "reference", "metric": "scanned GB/s", "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sample / value / 1e6, "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": threads, "kind": "port",
                         "sample": (("the whole " if sample >= size - 512 else "the first ") + f"{sample / (1 << 30):.2f} GiB of the configured {args.gib:g} GiB text per step, "
                                    f"{threads} newline-aligned shards in parallel; oracle port = reference loop (gzgets split, per-line match, strcpy) "
                                    "with PCRE2-JIT standing in for Hyperscan (vs PCRE2 proxy, not vs Hyperscan)"),
                         "matched_lines_per_s": matches / (sample / value / 1e9)},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
class LineCollector:
    """hs_event callback that keeps the line numbers of every result (numpy view of the 24-byte result records)."""

    def __init__(self) -> None:
        import numpy as np  # pylint: disable=import-outside-toplevel

        self.np = np
        self.parts: list = []
        self.dtype = np.dtype([("id", "<u4"), ("pad", "<u4"), ("line_number", "<u8"), ("line", "<u8")])
        self.func = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int)(self._on_batch)

    def _on_batch(self, results, count) -> None:
        raw = (ctypes.c_ubyte * (24 * count)).from_address(results)
        self.parts.append(self.np.frombuffer(raw, dtype=self.dtype, count=count)["line_number"].copy())

    def lines(self):
        return self.np.concatenate(self.parts) if self.parts else self.np.empty(0, dtype=self.np.uint64)


DUMP_BYTES = 64 << 20


def dump_outputs(directory: str, prefix: str, last, scan_records) -> None:
    """Write what the last timed step computed (float64 .npy files, at most DUMP_BYTES in all):
      counts       : [bytes_scanned, lines, matches] of that step's statistics, what the timed call returns;
      line_numbers : the matched line numbers in delivery order, from one more pass of the same call over the same device
                     text with a callback (the timed call only counts them); a fixed seeded sample of them, kept in order,
                     when there are more than fit."""
    import numpy as np  # pylint: disable=import-outside-toplevel

    counts = np.array([last.bytes_scanned, last.lines, last.matches], dtype=np.float64)
    collector = LineCollector()
    scan_records(ctypes.cast(collector.func, ctypes.c_void_p))
    lines = collector.lines()
    assert lines.size == last.matches, f"{lines.size} delivered records, the timed step counted {last.matches}"
    cap = (DUMP_BYTES - counts.nbytes) // 8
    if lines.size > cap:
        lines = lines[np.sort(np.random.default_rng(0).choice(lines.size, cap, replace=False))]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, f"{prefix}counts.npy"), counts)
    np.save(os.path.join(directory, f"{prefix}line_numbers.npy"), lines.astype(np.float64))


def main() -> None:  # pylint: disable=too-many-locals,too-many-statements,too-many-branches
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import numpy as np  # pylint: disable=import-outside-toplevel

    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    patterns = synth.C2_PATTERNS
    config = {"workload": WORKLOAD, "patterns": len(patterns), "line_bytes_mean": 151,
              "l2": "inputs (GiBs) are far larger than the 126 MB L2, no flush needed", "parallelism": f"shard{world}",
              "buffer_size": 262140}
    if args.strong:
        config["gib_total"] = args.gib
    else:
        config["gib_per_gpu"] = args.gib

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, config, patterns)
        return

    # ------------------------------------------------------------------ our arm
    import torch  # pylint: disable=import-outside-toplevel
    import torch.distributed as dist  # pylint: disable=import-outside-toplevel

    from gpu_api import Stats  # pylint: disable=import-outside-toplevel
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = utils._get_hyperscanner_lib()  # pylint: disable=protected-access
    lib.gpugrep_set_device(local_rank)
    lib.gpugrep_last_error.restype = ctypes.c_char_p
    lib.gpugrep_scan_buffer.argtypes = [
        ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p,
    ]
    discard = ctypes.cast(lib.gpugrep_discard_results, ctypes.c_void_p)
    pa, fa, ia, npat = marshal(patterns)

    # ---- the corpus of this rank
    total_size = int(args.gib * (1 << 30))
    if args.strong:
        # block k of the global text comes from seed 1234 + k: rank r generates only its own blocks
        nblocks = (total_size + BLOCK - 1) // BLOCK
        first, last = nblocks * rank // world, nblocks * (rank + 1) // world
        size = min(total_size, last * BLOCK) - first * BLOCK
        seed = 1234 + first
    else:
        size, seed = total_size, 1234 + 1000 * rank
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    t0 = time.perf_counter()
    lines = synth.fill_syslog(host.numpy(), seed=seed)
    gen_s = time.perf_counter() - t0
    dev = host.cuda(non_blocking=False)
    torch.cuda.synchronize()
    # a dedicated (non-default) stream: the library enqueues every kernel of the device-resident passes on it, so the
    # CUDA events below bracket exactly the work that is timed
    stream = torch.cuda.Stream()

    def scan(ptr: int, nbytes: int, location: int, callback, pats=(pa, fa, ia, npat), batch: int = 4096) -> Stats:
        st = Stats()
        rc = lib.gpugrep_scan_buffer(ptr, nbytes, location, pats[0], pats[1], pats[2], pats[3], callback, 262140, batch, 0,
                                     ctypes.c_void_p(stream.cuda_stream) if location == 1 else None, ctypes.byref(st))
        if rc != 0:
            raise RuntimeError(f"gpugrep_scan_buffer failed with code {rc}: {lib.gpugrep_last_error()}")
        return st

    def barrier() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(value: float, op) -> float:
        if world == 1:
            return value
        t = torch.tensor([value], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(value: float) -> float:
        return reduce(value, dist.ReduceOp.MAX)

    def sum_over_ranks(value: float) -> float:
        return reduce(value, dist.ReduceOp.SUM)

    # ---- device-resident: value + roofline
    sampler = ClockSampler(local_rank)
    if rank == 0:   # one poller per box is enough: the ranks share the host
        sampler.start()
        sampler.wait_first()
    for _ in range(args.warmup):
        scan(dev.data_ptr(), size, 1, None)
    barrier()
    window_begin = time.perf_counter()
    begin, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = stream_launches = 0
    stream_ms = gpu_ms = 0.0
    matches = candidates = 0
    stream.wait_stream(torch.cuda.current_stream())
    begin.record(stream)
    st = None
    for _ in range(args.steps):
        st = scan(dev.data_ptr(), size, 1, None)
        launches += st.launches
        stream_launches += st.stream_launches
        stream_ms += st.stream_kernel_ms
        gpu_ms += st.gpu_ms
        matches, candidates = st.matches, st.candidates
    end.record(stream)
    barrier()
    sampler.windows.append((window_begin, time.perf_counter()))
    if args.dump_outputs and st is not None:
        dump_outputs(args.dump_outputs, f"rank{rank}_" if world > 1 else "", st,
                     lambda callback: scan(dev.data_ptr(), size, 1, callback))
    dev_ms = max_over_ranks(begin.elapsed_time(end))
    total_bytes = sum_over_ranks(float(size))
    value = total_bytes * args.steps / (dev_ms / 1e3) / 1e9
    total_matches = sum_over_ranks(float(matches))

    # ---- end to end from pinned host memory through the C ABI (H2D + kernels + D2H + delivery)
    for _ in range(max(1, args.warmup // 2)):
        scan(host.data_ptr(), size, 0, discard)
    barrier()
    t0 = time.perf_counter()
    h2d = d2h = 0
    for _ in range(args.steps):
        st = scan(host.data_ptr(), size, 0, discard)
        h2d, d2h = st.h2d_bytes, st.d2h_bytes
    barrier()
    e2e_local = time.perf_counter() - t0
    sampler.windows.append((t0, t0 + e2e_local))
    clocks = sampler.stop() if rank == 0 else None   # samples of both timed regions
    e2e_s = max_over_ranks(e2e_local)
    e2e_value = total_bytes * args.steps / e2e_s / 1e9
    h2d_total, d2h_total = sum_over_ranks(float(h2d)), sum_over_ranks(float(d2h))

    # ---- strong scaling: merge of the shard results, checked against a single-GPU pass of the whole text
    merge = None
    if args.strong:
        collector = LineCollector()
        st = scan(host.data_ptr(), size, 0, ctypes.cast(collector.func, ctypes.c_void_p))
        mine = collector.lines().astype(np.int64)
        counts = torch.tensor([int(st.lines), int(mine.size)], dtype=torch.int64, device="cuda")
        gathered = [torch.zeros_like(counts) for _ in range(world)]
        if world > 1:
            dist.all_gather(gathered, counts)   # the only exchange: line and match counts of the shards
        else:
            gathered = [counts]
        table = [tuple(int(v) for v in g.tolist()) for g in gathered]
        line_base = sum(t[0] for t in table[:rank])
        rebased = torch.from_numpy(mine + line_base).cuda()
        longest = max(t[1] for t in table)
        padded = torch.full((max(1, longest),), -1, dtype=torch.int64, device="cuda")
        padded[: rebased.numel()] = rebased
        parts = [torch.empty_like(padded) for _ in range(world)] if rank == 0 else None
        if world > 1:
            dist.gather(padded, parts, dst=0)
        else:
            parts = [padded]
        if rank == 0:
            merged = np.concatenate([parts[r][: table[r][1]].cpu().numpy() for r in range(world)])
            whole = torch.empty(total_size, dtype=torch.uint8).pin_memory()
            synth.fill_syslog(whole.numpy(), seed=1234)
            single = LineCollector()
            scan(whole.data_ptr(), total_size, 0, ctypes.cast(single.func, ctypes.c_void_p))
            expected = single.lines().astype(np.int64)
            merge = {"shards": world, "merged_records": int(merged.size), "single_gpu_records": int(expected.size),
                     "identical": bool(merged.size == expected.size and np.array_equal(merged, expected)),
                     "exchange": "all_gather of (lines, matches) per shard; records gathered to rank 0 only for this check"}
            del whole
        barrier()

    peak, peak_source = load_peaks()
    per_step_launches = max(1, stream_launches // max(1, args.steps))
    kernel_bytes = size / per_step_launches   # algorithmic bytes per k_stream launch
    avg_launch_ms = stream_ms / max(1, stream_launches)
    achieved = kernel_bytes / (avg_launch_ms / 1e3) / 1e9 if avg_launch_ms > 0 else 0.0

    # ---- the other BASELINE configurations on N GPUs: every rank scans its own copy of the text (weak scaling, like the
    # headline), time = max over ranks.  One gather at the end, also when a rank failed, so that no rank waits for another.
    multi_extra = None
    if world > 1 and not args.no_extras and not args.strong:
        local = torch.full((len(DEVICE_LEGS), 3), float("nan"), dtype=torch.float64)
        try:
            legs = device_legs(lib, scan, host, dev, size, stream, reuse_host=True)
            for k, name in enumerate(DEVICE_LEGS):
                local[k] = torch.tensor([legs[name]["ms"], legs[name]["bytes"], legs[name]["matches"]], dtype=torch.float64)
        except Exception as error:  # pylint: disable=broad-except
            print(f"rank {rank}: extra legs failed: {error}", file=sys.stderr)
        gathered = [torch.empty_like(local, device=dev.device) for _ in range(world)]
        dist.all_gather(gathered, local.to(dev.device))
        if rank == 0:
            stacked = torch.stack([g.cpu() for g in gathered])   # [rank][leg][ms, bytes, matches]
            multi_extra = {}
            for k, name in enumerate(DEVICE_LEGS):
                ms, nbytes, matches = stacked[:, k, 0], stacked[:, k, 1], stacked[:, k, 2]
                if bool(torch.isnan(ms).any()):
                    multi_extra[name] = {"value": None, "failed_ranks": [int(r) for r in torch.nonzero(torch.isnan(ms)).flatten()]}
                    continue
                multi_extra[name] = {"value": float(nbytes.sum() / ms.max() / 1e6), "unit": "GB/s", "n_gpus": world, "bytes_per_gpu": int(nbytes[0]),
                                     "ms_max_over_ranks": float(ms.max()), "ms_min_over_ranks": float(ms.min()),
                                     "matches": int(matches.sum())}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    line = {
        "metric": "scanned GB/s", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "config": config,
        "matched_lines_per_s": total_matches * args.steps / (dev_ms / 1e3),
        "matched_lines_per_step": total_matches, "lines_per_step": float(lines) if world == 1 else None,
        "candidates_per_gib": candidates / (size / (1 << 30)),
        "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": int(d2h_total),
                "ms_per_step": e2e_s * 1e3 / args.steps, "source": "pinned host memory -> gpugrep_scan_buffer (C ABI) -> native discard callback"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "kernel": "k_stream (newline count + literal prefilter)", "peak_source": peak_source,
                     "algorithmic_bytes_per_launch": kernel_bytes, "avg_launch_ms": avg_launch_ms,
                     "kernel_share_of_gpu_time": stream_ms / gpu_ms if gpu_ms else None,
                     "whole_pipeline_frac": (size * args.steps / (gpu_ms / 1e3) / 1e9) / peak if gpu_ms else None,
                     "value_frac_of_peak": value / world / peak},
        "clocks": clocks,
        "corpus_generation_s": gen_s,
    }
    if merge is not None:
        line["merge_check"] = merge
    if multi_extra is not None:
        line["extra"] = multi_extra
    # DRAM traffic of the roofline kernel from the committed ncu capture (profiles/), scaled to this run's launch size
    for name in ("r2_k_stream_traffic.json", "r1_k_stream_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name), encoding="utf-8") as handle:
                cap = json.load(handle)
            line["roofline"]["traffic"] = (cap["dram_bytes_read"] + cap["dram_bytes_write"]) * kernel_bytes / cap["launch_bytes"]
            line["roofline"]["traffic_source"] = cap["source"]
            break
        except (OSError, KeyError, ValueError):
            continue

    if world == 1 and not args.strong:
        view = host.numpy()
        oracle = None
        try:
            oracle = load_oracle()
        except Exception as error:  # pylint: disable=broad-except
            line["parity"] = {"checked": False, "error": str(error)}
        # ---- parity of what was timed: line numbers of a bounded prefix, GPU vs oracle on all host cores
        if oracle is not None:
            try:
                threads = os.cpu_count() or 1
                gbs, _, _, _ = oracle_throughput(oracle, view, size, patterns, threads, 2.0)
                sample = min(size, int(gbs * 1e9 * 12.0))   # about 12 s of oracle time
                while sample > 1 and view[sample - 1] != 10:
                    sample -= 1
                secs, cpu_matches, cpu_lines = oracle_scan(oracle, view, sample, patterns, threads, True)
                collector = LineCollector()
                scan(host.data_ptr(), sample, 0, ctypes.cast(collector.func, ctypes.c_void_p))   # the e2e path: same kernels, lines gathered from pinned memory
                gpu_lines = collector.lines()
                st_dev = scan(dev.data_ptr(), sample, 1, None)   # the device-resident path counts the same lines
                assert int(st_dev.matches) == int(gpu_lines.size), "device-resident count differs from the delivered records"
                same = bool(gpu_lines.size == cpu_lines.size and np.array_equal(gpu_lines, cpu_lines))
                line["parity"] = {"checked": True, "identical": same, "parity_checked_bytes": int(sample), "matched_lines": int(cpu_matches),
                                  "gpu_matched_lines": int(gpu_lines.size), "oracle_seconds": secs, "oracle_threads": threads,
                                  "what": "every matched line number of the first parity_checked_bytes of the timed text, in delivery order"}
                if not same:
                    raise AssertionError("GPU result differs from the oracle on the benchmarked text")
            except AssertionError:
                print(json.dumps(line))
                raise
            except Exception as error:  # pylint: disable=broad-except
                line["parity"] = {"checked": False, "error": str(error)}
        # ---- the reference-facing call itself: hyperscan(path) on a file in tmpfs, and the Python layer on top of it
        shm = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
        path = os.path.join(shm, f"gpugrep_bench_{os.getpid()}.log")
        try:
            file_bytes = min(size, 4 << 30)
            while file_bytes > 1 and view[file_bytes - 1] != 10:
                file_bytes -= 1
            view[:file_bytes].tofile(path)
            lib.gpugrep_scan_file.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p]
            fst = Stats()
            file_s = 0.0
            for _ in range(3):
                t0 = time.perf_counter()
                rc = lib.gpugrep_scan_file(path.encode(), pa, fa, ia, npat, discard, 262140, 4096, 0, ctypes.byref(fst))
                file_s = time.perf_counter() - t0
                assert rc == 0
            line["e2e_file"] = {"value": file_bytes / file_s / 1e9, "unit": "GB/s", "bytes": file_bytes, "matches": int(fst.matches),
                                "source": "hyperscan(path)-equivalent gpugrep_scan_file on a tmpfs file, native discard callback, third of 3 runs"}
            if not args.no_extras:
                import hypergrep_b200 as hg  # pylint: disable=import-outside-toplevel

                t0 = time.perf_counter()
                count, code = hg.grep(path, patterns, count_only=True)
                grep_s = time.perf_counter() - t0
                seen = [0]

                def on_match(_matches, count_):   # the default 16-slot batches of the reference API: one Python frame per batch
                    seen[0] += count_

                t0 = time.perf_counter()
                code2 = hg.scan(path, patterns, on_match)
                scan_s = time.perf_counter() - t0
                line["e2e_python"] = {
                    "grep_count_only": {"value": file_bytes / grep_s / 1e9, "unit": "GB/s", "matches": int(count), "rc": int(code)},
                    "scan_python_callback_16": {"value": file_bytes / scan_s / 1e9, "unit": "GB/s", "matches": int(seen[0]), "rc": int(code2),
                                                "matched_lines_per_s": seen[0] / scan_s},
                    "bytes": file_bytes, "source": "hypergrep_b200.grep(path, patterns, count_only=True) and hypergrep_b200.scan(path, patterns, "
                                                   "python_callback) with the default buffer_count=16, tmpfs file"}
        except Exception as error:  # pylint: disable=broad-except
            line.setdefault("e2e_file", {"value": None, "error": str(error)})
        finally:
            if os.path.exists(path):
                os.unlink(path)
        # ---- the other BASELINE configurations (device-resident, 2 GiB of the same text unless stated)
        if not args.no_extras:
            try:
                line["extra"] = extra_configs(lib, scan, host, dev, size, stream)
            except Exception as error:  # pylint: disable=broad-except
                line["extra"] = {"error": str(error)}
        # ---- CPU baseline (one core)
        if oracle is not None:
            try:
                gbs, sample, cpu_matches, secs = oracle_throughput(oracle, view, size, patterns, 1, args.cpu_seconds)
                line["cpu_baseline"] = {
                    "value": gbs, "unit": "GB/s", "cores": 1, "kind": "port",
                    "sample": f"first {sample / (1 << 20):.0f} MiB of the same text, {secs:.1f} s; oracle port = reference loop shape with "
                              "PCRE2-JIT standing in for Hyperscan (not installable here): a PCRE2 proxy, not Hyperscan",
                    "matched_lines_per_s": cpu_matches / secs, "host_cores_available": os.cpu_count()}
            except Exception as error:  # pylint: disable=broad-except
                line["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": 1, "kind": "port", "sample": f"failed: {error}"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def device_legs(lib, scan, host, dev, size: int, stream, reuse_host: bool = False, oracle=None) -> dict:  # pylint: disable=too-many-locals
    """Device-resident throughput of BASELINE configs[0], [2] and [4] on this rank's GPU.  `reuse_host`: the pinned text of
    the headline run is no longer needed (multi-rank runs) and serves as the staging buffer, so that eight ranks do not pin
    another 3 GiB each."""
    import numpy as np  # pylint: disable=import-outside-toplevel
    import torch  # pylint: disable=import-outside-toplevel

    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    out: dict = {}
    part = min(size, 2 << 30)
    view = host.numpy()
    while part > 1 and view[part - 1] != 10:
        part -= 1

    def timed(ptr: int, nbytes: int, pats, passes: int = 3):
        st = None
        begin, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(passes):
            if k == passes - 1:
                begin.record(stream)
            t0 = time.perf_counter()
            st = scan(ptr, nbytes, 1, None, pats)
            if os.environ.get("GPUGREP_BENCH_TRACE"):
                print(f"trace pass {k}: wall {1e3 * (time.perf_counter() - t0):.3f} ms, gpu {st.gpu_ms:.3f} ms, stream {st.stream_kernel_ms:.3f} ms, launches {st.launches}", file=sys.stderr)
        end.record(stream)
        torch.cuda.synchronize()
        ms = begin.elapsed_time(end)
        return {"value": nbytes / ms / 1e6, "unit": "GB/s", "bytes": nbytes, "matches": int(st.matches), "ms": ms, "kernel_ms": st.gpu_ms, "stream_kernel_ms": st.stream_kernel_ms,
                "candidates_per_gib": st.candidates / (nbytes / (1 << 30)), "path": int(st.path), "launches": int(st.launches),
                "segments": int(st.segments), "split_segments": int(st.split_segments)}

    def parity(text_view, text_ptr: int, nbytes: int, pat_list, flags, marshaled, sample_bytes: int) -> dict:
        """Matched line numbers of a prefix of the leg's text: library (host path, records delivered) against the oracle on all
        host cores.  The device-resident pass that was timed counts the same text (its `matches` are for the whole of it)."""
        sample = min(nbytes, sample_bytes)
        while sample > 1 and text_view[sample - 1] != 10:
            sample -= 1
        threads = os.cpu_count() or 1
        secs, cpu_matches, cpu_lines = oracle_scan(oracle, text_view, sample, pat_list, threads, True, flags)
        collector = LineCollector()
        scan(text_ptr, sample, 0, ctypes.cast(collector.func, ctypes.c_void_p), marshaled)
        gpu_lines = collector.lines()
        same = bool(gpu_lines.size == cpu_lines.size and np.array_equal(gpu_lines, cpu_lines))
        if not same:
            print(f"PARITY FAILURE in an extra leg: {gpu_lines.size} lines, oracle {cpu_lines.size}", file=sys.stderr)
        return {"checked": True, "identical": same, "parity_checked_bytes": int(sample), "matched_lines": int(cpu_matches),
                "gpu_matched_lines": int(gpu_lines.size), "oracle_seconds": secs, "oracle_threads": threads}

    def with_parity(result: dict, *args) -> dict:
        if oracle is not None:
            try:
                result["parity"] = parity(*args)
            except Exception as error:  # pylint: disable=broad-except
                result["parity"] = {"checked": False, "error": str(error)}
        return result

    c1 = marshal(synth.C1_PATTERNS)
    out["configs[0] 'ERROR' (1 literal)"] = with_parity(timed(dev.data_ptr(), part, c1), view, host.data_ptr(), part, synth.C1_PATTERNS, None, c1, part)
    c3, plants = synth.c3_patterns()
    planted = host[:part] if reuse_host else torch.empty(part, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(planted.numpy(), seed=4321, plants=plants, plant_ppm=1000)
    planted_dev = planted.cuda()
    c3m = marshal(c3)
    out["configs[2] 1,000 IOC patterns"] = with_parity(timed(planted_dev.data_ptr(), part, c3m), planted.numpy(), planted.data_ptr(), part, c3, None, c3m,
                                                        64 << 20)   # (the PCRE2 proxy takes ~0.1 s per MiB of this set on 16 cores)
    del planted_dev, planted
    # configs[4]: caseless template patterns over long JSON-ish lines (an 8 MiB generated sample, tiled to 1 GiB)
    c5 = synth.c5_patterns(10000)
    sample = np.frombuffer(synth.jsonish_bytes(8 << 20, patterns_to_plant=["session_4242 failed", "code=E31337abcd"]), dtype=np.uint8)
    long_size = 1 << 30
    if reuse_host and host.numel() >= long_size:
        tiled = host[:long_size]
        tiled.numpy()[:] = np.tile(sample, -(-long_size // sample.size))[:long_size]
    else:
        tiled = torch.from_numpy(np.tile(sample, -(-long_size // sample.size))[:long_size].copy())
    tiled[-1] = 10
    tiled_dev = tiled.cuda()
    c5m = marshal(c5, [15] * len(c5))
    out["configs[4] 10,000 caseless patterns, 2-16 KiB lines"] = with_parity(timed(tiled_dev.data_ptr(), long_size, c5m, passes=2), tiled.numpy(),
                                                                              tiled.data_ptr(), long_size, c5, [15] * len(c5), c5m, 24 << 20)
    del tiled_dev, tiled
    return out


DEVICE_LEGS = ["configs[0] 'ERROR' (1 literal)", "configs[2] 1,000 IOC patterns", "configs[4] 10,000 caseless patterns, 2-16 KiB lines"]


def extra_configs(lib, scan, host, dev, size: int, stream) -> dict:
    """The other BASELINE configurations: device-resident C1 / C3 / C5 (device_legs) and the C4 file legs."""
    import hypergrep_b200.multiscanner as multiscanner  # pylint: disable=import-outside-toplevel

    oracle = None
    try:
        oracle = load_oracle()
    except Exception:  # pylint: disable=broad-except
        pass
    out = device_legs(lib, scan, host, dev, size, stream, oracle=oracle)
    view = host.numpy()
    # configs[3] shape: files (plain / gzip -6 / zstd -3) through the reference-facing CLI entry, one job per file
    try:
        out["configs[3] files through multiscanner.parallel_grep"] = file_leg(view, multiscanner)
    except Exception as error:  # pylint: disable=broad-except
        out["configs[3] files through multiscanner.parallel_grep"] = {"error": str(error)}
    return out


def file_leg(view, multiscanner) -> dict:
    """8 files x 64 MiB of the text as plain / gzip / zstd copies in tmpfs through multiscanner.parallel_grep (count per
    file, C2 patterns).  GB/s of decompressed text; the decoders run on host threads (stated ingest, not the hot path)."""
    import contextlib  # pylint: disable=import-outside-toplevel
    import gzip  # pylint: disable=import-outside-toplevel
    import io  # pylint: disable=import-outside-toplevel
    import tempfile  # pylint: disable=import-outside-toplevel
    from concurrent.futures import ThreadPoolExecutor  # pylint: disable=import-outside-toplevel

    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    files, each = 8, 64 << 20
    zstd = ctypes.CDLL("libzstd.so.1")
    zstd.ZSTD_compressBound.restype = ctypes.c_size_t
    zstd.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    zstd.ZSTD_compress.restype = ctypes.c_size_t
    zstd.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else None
    result: dict = {"files": files, "bytes_per_file": each, "host_threads": min(files, max(1, (os.cpu_count() or 2) - 1))}
    with tempfile.TemporaryDirectory(dir=shm) as tmp:
        chunks = []
        for k in range(files):
            end = (k + 1) * each
            while end > 1 and view[end - 1] != 10:
                end -= 1
            chunks.append(view[k * each:end].tobytes())

        def write(kind: str, k: int) -> str:
            path = os.path.join(tmp, f"part{k}.log" + {"plain": "", "gzip": ".gz", "zstd": ".zst"}[kind])
            data = chunks[k]
            if kind == "gzip":
                data = gzip.compress(data, 6)
            elif kind == "zstd":
                bound = zstd.ZSTD_compressBound(len(data))
                buf = ctypes.create_string_buffer(bound)
                n = zstd.ZSTD_compress(buf, bound, data, len(data), 3)
                data = buf.raw[:n]
            with open(path, "wb") as handle:
                handle.write(data)
            return path

        total = sum(len(c) for c in chunks)
        for kind in ("plain", "zstd", "gzip"):
            with ThreadPoolExecutor(max_workers=8) as pool:
                paths = list(pool.map(lambda k, kind=kind: write(kind, k), range(files)))
            compressed = sum(os.path.getsize(p) for p in paths)
            best = None
            for _ in range(5 if kind == "plain" else 2):   # (eight scans at once warm their pinned slots up over the first runs)
                sink = io.StringIO()
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(sink):
                    code = multiscanner.parallel_grep(paths, synth.C2_PATTERNS, count_results=True, total_results=True)
                elapsed = time.perf_counter() - t0
                best = elapsed if best is None else min(best, elapsed)
            result[kind] = {"value": total / best / 1e9, "unit": "GB/s of text", "seconds": best, "compression_ratio": total / compressed,
                            "rc": int(code), "output_tail": sink.getvalue().strip().splitlines()[-1:]}
            for p in paths:
                os.unlink(p)

        # ONE compressed file of 256 MiB of text: a single member / frame (what `gzip` and `zstd` write: one decode thread,
        # like the reference's gzgets() stream) against many members / frames (bgzip, pzstd, concatenated rotations: decoded
        # by helper threads ahead of the reader, hypergrep_b200/csrc/ingest_members.cpp).
        text = b"".join(chunks[:4])
        cores = os.cpu_count() or 2
        single: dict = {"bytes": len(text), "decode_threads_many": 1 + max(0, min(16, cores - 2))}

        def pieces(step: int) -> list:
            out, at = [], 0
            while at < len(text):
                end = text.find(b"\n", min(len(text) - 1, at + step)) + 1 or len(text)
                out.append(text[at:end])
                at = end
            return out

        def zstd_frame(data: bytes) -> bytes:
            bound = zstd.ZSTD_compressBound(len(data))
            buf = ctypes.create_string_buffer(bound)
            written = zstd.ZSTD_compress(buf, bound, data, len(data), 3)
            return buf.raw[:written]

        layouts = {
            "zstd_one_frame": (".zst", zstd_frame, [text]),
            "zstd_frames_8MiB": (".zst", zstd_frame, pieces(8 << 20)),
            "gzip_one_member": (".gz", lambda d: gzip.compress(d, 1), [text]),
            "gzip_members_1MiB": (".gz", lambda d: gzip.compress(d, 1), pieces(1 << 20)),
        }
        for name, (suffix, pack, parts) in layouts.items():
            path = os.path.join(tmp, "single.log" + suffix)
            with ThreadPoolExecutor(max_workers=max(1, min(16, cores - 1))) as pool:
                blob = b"".join(pool.map(pack, parts))
            with open(path, "wb") as handle:
                handle.write(blob)
            best, counts = None, set()
            for _ in range(2):
                sink = io.StringIO()
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(sink):
                    code = multiscanner.parallel_grep([path], synth.C2_PATTERNS, count_results=True)
                elapsed = time.perf_counter() - t0
                best = elapsed if best is None else min(best, elapsed)
                counts.add(sink.getvalue().strip())
            single[name] = {"value": len(text) / best / 1e9, "unit": "GB/s of text", "seconds": best, "members": len(parts),
                            "compression_ratio": len(text) / len(blob), "rc": int(code), "output": sorted(counts)}
            os.unlink(path)
        # the same text must give the same count in every layout
        single["counts_agree"] = len({tuple(o.split(":")[-1] for o in single[n]["output"]) for n in layouts}) == 1
        result["single_file"] = single
    return result


if __name__ == "__main__":
    main()
