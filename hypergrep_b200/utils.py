"""Host-side mirror of the reference's ctypes layer (reference hypergrep/utils.py), bound to libgpugrep.so.

Same names, argument meaning, defaults and error behaviour as the reference so that its tests read the same
against this package; only the native library underneath changes.  All regex and line work happens in the
CUDA engine: there is no Python/CPU matching fallback, and loading fails loudly if the library is missing.
"""

from __future__ import annotations

import bisect
import ctypes
import itertools
import os
import re
import threading
from typing import Callable, Sequence

# hs_compile.h flag bits forwarded to the engine (reference utils.py:9-13).
HS_FLAG_CASELESS = 1
HS_FLAG_DOTALL = 2
HS_FLAG_MULTILINE = 4
HS_FLAG_SINGLEMATCH = 8
_DEFAULT_FLAGS = HS_FLAG_DOTALL | HS_FLAG_MULTILINE | HS_FLAG_SINGLEMATCH

# 101-125 are reserved for this layer (reference utils.py:15-16).
RC_INVALID_FILE = 101
_RC_INTERRUPTED = 130

# Result.id of a context line (scan()/grep() with before_context / after_context; GPUGREP_CONTEXT_ID in include/gpugrep.h).
CONTEXT_ID = 0xFFFFFFFF

_LIB_NAME = "libgpugrep.so"
_lock = threading.Lock()
_state: dict = {"lib": None, "libzstd": None, "libhs": None}


class Result(ctypes.Structure):
    """One matched line as delivered by the engine: 24-byte record (reference hyperscanner.c:42-46, utils.py:25-40).

    ``line`` points at engine-owned, NUL-terminated bytes that are only valid during the callback.
    """

    _fields_ = [
        ("id", ctypes.c_uint),
        ("line_number", ctypes.c_ulonglong),
        ("line", ctypes.c_char_p),
    ]


# void (*hs_event)(hyperscanner_result_t*, int)  (reference hyperscanner.c:54, utils.py:45-51)
CALLBACK_TYPE = ctypes.CFUNCTYPE(None, ctypes.POINTER(Result), ctypes.c_int)


def _library_path() -> str:
    override = os.environ.get("GPUGREP_LIBRARY")
    if override:
        return override
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", _LIB_NAME)


def _get_hyperscanner_lib() -> ctypes.CDLL:
    """Load libgpugrep.so once per process (lazily, so forked pool workers can load it themselves).

    Same role and name as reference utils.py:67-81.  No CUDA context is created by loading or by
    ``check_patterns``; the engine initialises CUDA inside the first ``hyperscan`` call.
    """
    with _lock:
        if _state["lib"] is None:
            path = _library_path()
            if not os.path.exists(path):
                raise OSError(
                    f"{path}: native engine not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "or `make -C hypergrep_b200/csrc`; there is no CPU fallback."
                )
            lib = ctypes.CDLL(path)
            if _state["libzstd"]:
                lib.gpugrep_set_zstd_path.argtypes = [ctypes.c_char_p]
                lib.gpugrep_set_zstd_path(_state["libzstd"].encode())
            _state["lib"] = lib
        return _state["lib"]


def configure_libraries(libhs: str | None = None, libzstd: str | None = None) -> None:
    """Accept the reference's library overrides (reference utils.py:125-144).

    ``libhs`` is recorded and otherwise ignored: no Hyperscan is involved.  ``libzstd`` names the shared
    object the engine dlopen()s for .zst ingest (default: the system libzstd.so.1).  As in the reference,
    calling this after the native library is in use is an error.
    """
    if libhs:
        if _state["lib"] is not None:
            raise ValueError("libhs already loaded, configuration overrides must be called before library usage")
        _state["libhs"] = libhs
    if libzstd:
        if _state["lib"] is not None:
            raise ValueError("libzstd already loaded, configuration overrides must be called before library usage")
        _state["libzstd"] = libzstd


def prepare_patterns(
    patterns: Sequence[str],
    flags: Sequence[int] = (),
    ids: Sequence[int] = (),
) -> tuple[ctypes.Array, ctypes.Array, ctypes.Array]:
    """Marshal patterns, flags and ids into the C arrays of the boundary (reference utils.py:234-289).

    Defaults: flags DOTALL|MULTILINE|SINGLEMATCH for every pattern, ids all 0 (one report per line).
    Raises ValueError for length mismatches and for empty patterns, like the reference.
    """
    count = len(patterns)
    if not flags:
        flags = [_DEFAULT_FLAGS] * count
    if len(flags) != count:
        raise ValueError(
            f"Found {len(flags)} flags, expecting {count}. Hyperscan flags must be provided for each regex to compile the database."
        )
    if not ids:
        ids = [0] * count
    if len(ids) != count:
        raise ValueError(
            f"Found {len(ids)} ids, expecting {count}. Hyperscan ids must be provided for each regex to compile the database."
        )
    raw = []
    for pattern in patterns:
        if not pattern:
            raise ValueError(f'Invalid pattern "{pattern}" found. Please provide a valid regex for Intel Hyperscan.')
        raw.append(pattern.encode())
    pattern_array = (ctypes.c_char_p * count)(*raw)
    flags_array = (ctypes.c_uint * count)(*[int(flag) for flag in flags])
    ids_array = (ctypes.c_uint * count)(*[int(id_num) for id_num in ids])
    return pattern_array, flags_array, ids_array


def check_compatibility(patterns: list, flags: Sequence[int] = (), fixed_strings: bool = False) -> int:
    """Compile-check patterns without scanning (reference utils.py:97-122): 0, or 4 when any pattern is rejected.
    ``fixed_strings``: the patterns are literals (``grep -F``), checked by gpugrep_check_literals."""
    pattern_array, flags_array, ids_array = prepare_patterns(patterns, flags=flags)
    lib = _get_hyperscanner_lib()
    if fixed_strings:
        return _literal_check_entry(lib)(pattern_array, flags_array, len(pattern_array))
    return lib.check_patterns(pattern_array, flags_array, ids_array, len(pattern_array))


_GREP_BATCH = 4096   # results per callback when grep() collects lines (the reference's scan() default is 16)


def scan(  # pylint: disable=too-many-arguments
    path: str,
    patterns: Sequence[str],
    callback: Callable,
    flags: Sequence[int] = (),
    ids: Sequence[int] = (),
    buffer_size: int = 262140,
    buffer_count: int = 16,
    max_match_count: int = 0,
    invert_match: bool = False,
    before_context: int = 0,
    after_context: int = 0,
    fixed_strings: bool = False,
) -> int:
    """Scan one plain/gzip/zstd file on the GPU, delivering matched lines in batches (reference utils.py:292-358).

    ``callback(matches, count)`` receives up to ``buffer_count`` ``Result`` records per call, in file order,
    with 0-based ``line_number``.  Returns the engine's code: 0, or 1-7 (reference hyperscanner.c:25-33).
    ``invert_match`` (``grep -v``) delivers the lines that no pattern matches instead, each with id 0, and
    ``max_match_count`` then counts those lines.
    ``before_context`` / ``after_context`` (``grep -B`` / ``-A``) also deliver the lines that lie up to that many lines
    before / after a selected line, with id ``CONTEXT_ID``; selected lines then carry id 0.  ``max_match_count`` counts
    selected lines, and the ``after_context`` lines behind the one that reaches it are still delivered, as context.
    ``fixed_strings`` (``grep -F``): the patterns are literals, not regular expressions (gpugrep_literal_scan_file); only
    ``HS_FLAG_CASELESS`` of the flags changes anything, and every record has id 0, so ``ids`` raise ValueError.
    """
    _check_context(before_context, after_context)
    if fixed_strings and ids:
        raise ValueError("fixed_strings scans take no ids: every selected line is reported with id 0")
    pattern_array, flags_array, ids_array = prepare_patterns(patterns, flags=flags, ids=ids)
    c_callback = CALLBACK_TYPE(callback)
    lib = _get_hyperscanner_lib()
    context = before_context > 0 or after_context > 0
    if fixed_strings:
        entry = _literal_entry(lib)
    else:
        entry = _context_entry(lib) if context else (_invert_entry(lib) if invert_match else None)
    outcome = {"rc": 0}

    def _run() -> None:
        if fixed_strings:
            outcome["rc"] = entry(path.encode(), pattern_array, flags_array, len(pattern_array), c_callback, buffer_size, buffer_count,
                                  max_match_count, before_context, after_context, int(invert_match), None)
            return
        if context:
            outcome["rc"] = entry(path.encode(), pattern_array, flags_array, ids_array, len(pattern_array), c_callback, buffer_size,
                                  buffer_count, max_match_count, before_context, after_context, int(invert_match), None)
            return
        if entry is not None:
            outcome["rc"] = entry(path.encode(), pattern_array, flags_array, ids_array, len(pattern_array), c_callback, buffer_size,
                                  buffer_count, max_match_count, None)
            return
        outcome["rc"] = lib.hyperscan(
            path.encode(),
            pattern_array,
            flags_array,
            ids_array,
            len(pattern_array),
            c_callback,
            buffer_size,
            buffer_count,
            ctypes.c_ulonglong(max_match_count),
        )

    # A daemon worker keeps the main thread interruptible, exactly as the reference does (utils.py:335-357).
    worker = threading.Thread(target=_run, daemon=True)
    worker.start()
    try:
        worker.join(timeout=3600)
    except KeyboardInterrupt:
        outcome["rc"] = _RC_INTERRUPTED
    return outcome["rc"]


class _Stats(ctypes.Structure):
    """gpugrep_stats (include/gpugrep.h)."""

    _fields_ = [
        ("bytes_scanned", ctypes.c_ulonglong), ("lines", ctypes.c_ulonglong), ("matches", ctypes.c_ulonglong),
        ("candidates", ctypes.c_ulonglong), ("h2d_bytes", ctypes.c_ulonglong), ("d2h_bytes", ctypes.c_ulonglong),
        ("gpu_ms", ctypes.c_double), ("stream_kernel_ms", ctypes.c_double), ("wall_ms", ctypes.c_double),
        ("launches", ctypes.c_uint), ("stream_launches", ctypes.c_uint), ("segments", ctypes.c_uint), ("path", ctypes.c_uint),
        ("split_segments", ctypes.c_uint), ("nul_segments", ctypes.c_uint),
    ]


_FILE_ENTRY_ARGTYPES = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                        ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p]


def _invert_entry(lib: ctypes.CDLL):
    """gpugrep_invert_scan_file of the loaded library.  Inverted matching has no CPU fallback: a library without the entry
    point (a plain libhyperscanner.so through GPUGREP_LIBRARY) is an error."""
    try:
        entry = lib.gpugrep_invert_scan_file
    except AttributeError as error:
        raise NotImplementedError(
            "invert_match needs gpugrep_invert_scan_file, which the loaded native library does not export "
            f"({_library_path()}); there is no CPU fallback"
        ) from error
    entry.restype = ctypes.c_int
    entry.argtypes = _FILE_ENTRY_ARGTYPES
    return entry


def _check_context(before_context: int, after_context: int) -> None:
    if before_context < 0 or after_context < 0:
        raise ValueError(f"context line counts must not be negative (before_context={before_context}, after_context={after_context})")
    if before_context > 0xFFFFFFFF or after_context > 0xFFFFFFFF:
        raise ValueError("context line counts must fit in 32 bits")


def _context_entry(lib: ctypes.CDLL):
    """gpugrep_context_scan_file of the loaded library.  Context lines have no CPU fallback: a library without the entry
    point (a plain libhyperscanner.so through GPUGREP_LIBRARY) is an error."""
    try:
        entry = lib.gpugrep_context_scan_file
    except AttributeError as error:
        raise NotImplementedError(
            "before_context / after_context need gpugrep_context_scan_file, which the loaded native library does not export "
            f"({_library_path()}); there is no CPU fallback"
        ) from error
    entry.restype = ctypes.c_int
    entry.argtypes = _FILE_ENTRY_ARGTYPES[:9] + [ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
    return entry


def _literal_entry(lib: ctypes.CDLL):
    """gpugrep_literal_scan_file of the loaded library.  Fixed strings have no CPU fallback: a library without the entry
    point (a plain libhyperscanner.so through GPUGREP_LIBRARY) is an error."""
    try:
        entry = lib.gpugrep_literal_scan_file
    except AttributeError as error:
        raise NotImplementedError(
            "fixed_strings needs gpugrep_literal_scan_file, which the loaded native library does not export "
            f"({_library_path()}); there is no CPU fallback"
        ) from error
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                      ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
    return entry


def _literal_check_entry(lib: ctypes.CDLL):
    """gpugrep_check_literals of the loaded library (see _literal_entry)."""
    try:
        entry = lib.gpugrep_check_literals
    except AttributeError as error:
        raise NotImplementedError(
            f"fixed_strings needs gpugrep_check_literals, which the loaded native library does not export ({_library_path()})"
        ) from error
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint]
    return entry


def _count_matches(path: str, patterns: Sequence[str], flags: Sequence[int], max_match_count: int,
                   invert_match: bool = False, fixed_strings: bool = False) -> tuple[int, int] | None:
    """Count-only scan without a callback: the library counts on the device and copies no line back
    (gpugrep_scan_file with on_event = NULL).  Returns None if the loaded library has no such entry point (a plain
    libhyperscanner.so), in which case the caller counts through the callback like the reference does.
    ``invert_match`` counts the lines without a match (gpugrep_invert_scan_file); it has no such fallback, nor has
    ``fixed_strings`` (gpugrep_literal_scan_file)."""
    lib = _get_hyperscanner_lib()
    if fixed_strings:
        entry = _literal_entry(lib)
    elif invert_match:
        entry = _invert_entry(lib)
    else:
        try:
            entry = lib.gpugrep_scan_file
        except AttributeError:
            return None
        entry.restype = ctypes.c_int
        entry.argtypes = _FILE_ENTRY_ARGTYPES
    pattern_array, flags_array, ids_array = prepare_patterns(patterns, flags=flags)
    stats = _Stats()
    outcome = {"rc": 0}

    def _run() -> None:
        if fixed_strings:
            outcome["rc"] = entry(path.encode(), pattern_array, flags_array, len(pattern_array), None, 262140, 16, max_match_count, 0, 0,
                                  int(invert_match), ctypes.byref(stats))
            return
        outcome["rc"] = entry(path.encode(), pattern_array, flags_array, ids_array, len(pattern_array), None, 262140, 16,
                              max_match_count, ctypes.byref(stats))

    worker = threading.Thread(target=_run, daemon=True)   # same interruptible wait as scan()
    worker.start()
    try:
        worker.join(timeout=3600)
    except KeyboardInterrupt:
        return 0, _RC_INTERRUPTED
    return int(stats.matches), outcome["rc"]


def grep(  # pylint: disable=too-many-arguments
    file: str,
    patterns: list[str],
    ignore_case: bool = False,
    count_only: bool = False,
    only_matching: bool = False,
    no_messages: bool = False,
    errors: str = "ignore",
    max_match_count: int = 0,
    invert_match: bool = False,
    before_context: int = 0,
    after_context: int = 0,
    fixed_strings: bool = False,
) -> tuple[int | list[tuple[int, str]] | list[tuple[int, str, bool]], int]:
    """grep-like collector on top of :func:`scan` (reference utils.py:147-231).

    Returns ``(results, return_code)`` where results is a count (``count_only``) or a list of
    ``(1-based line number, line text)``.  Missing files raise FileNotFoundError, directories ValueError,
    unless ``no_messages`` is set, in which case the code is RC_INVALID_FILE.
    ``invert_match`` (``grep -v``) selects the lines that no pattern matches; ``max_match_count`` and the count then
    refer to those lines, and ``only_matching`` gives ``[]`` (a line without a match has no matching parts).
    ``before_context`` / ``after_context`` (``grep -B`` / ``-A``) add the lines up to that many lines before / after each
    selected line; results are then ``(line number, line text, is_context)``.  ``count_only`` and ``only_matching`` ignore
    context.  Negative counts raise ValueError.
    ``fixed_strings`` (``grep -F``): the patterns are literals (:func:`scan`).  With ``only_matching`` the result is that of
    the ``re.escape``-d patterns as regular expressions.
    """
    _check_context(before_context, after_context)
    if fixed_strings and only_matching:
        patterns = [re.escape(pattern) for pattern in patterns]
        fixed_strings = False
    context = (before_context > 0 or after_context > 0) and not (count_only or only_matching)
    python_patterns = [] if fixed_strings else [re.compile(pattern) for pattern in patterns]
    collected: list[tuple[int, str]] = []
    counter = [0]

    code = 0
    if not os.path.exists(file):
        code = RC_INVALID_FILE
        if not no_messages:
            raise FileNotFoundError("No such file or directory")
    if os.path.isdir(file):
        code = RC_INVALID_FILE
        if not no_messages:
            raise ValueError("is a directory")
    if code:
        return (0 if count_only else collected), code
    if invert_match and only_matching and not count_only:
        return collected, code

    # `-o`: spans from the engine where that is exact (ASCII lines; patterns of one fixed width whose syntax means the same in
    # Python's re take the match END offsets, other patterns that pass the span screen the leftmost-first match spans),
    # re.finditer() as in the reference (utils.py:205-212) for everything else.
    widths = _span_widths(patterns) if only_matching else None
    exact = (_span_exact(patterns) or [False] * len(patterns)) if widths is not None else None
    groups: list[list[tuple[int, str]]] = []      # one entry per record (or per batch of span-route records), in record order
    deferred: list[tuple[int, int, bytes]] = []   # fixed-width route: (index into groups, pattern id, line bytes)
    span_lines = _SpanLines(widths, exact) if widths is not None else None

    def _on_batch(matches: ctypes.Array, count: int) -> None:
        if count_only:
            counter[0] += count
            return
        if span_lines is not None and span_lines.take_batch(matches, count, groups):
            return
        for position in range(count):
            record = matches[position]
            raw = record.line
            if only_matching:
                # Same quirk as the reference (utils.py:205-212): record.id is the user id, not the pattern index.
                if widths is not None and (widths[record.id] > 0 or exact[record.id]) and raw.isascii() and raw.endswith(b"\n"):
                    if widths[record.id] > 0:
                        deferred.append((len(groups), record.id, raw))
                        groups.append([(record.line_number + 1, "")])
                    else:
                        span_lines.add(record.id, [record.line_number], [raw], groups)
                    continue
                text = raw.decode(errors=errors)
                groups.append([(record.line_number + 1, f"{part.group()}\n") for part in python_patterns[record.id].finditer(text)])
            elif context:
                collected.append((record.line_number + 1, raw.decode(errors=errors), record.id == CONTEXT_ID))
            else:
                collected.append((record.line_number + 1, raw.decode(errors=errors)))

    pattern_flags = _DEFAULT_FLAGS | (HS_FLAG_CASELESS if ignore_case else 0)
    if count_only:
        # SURVEY.md section 8(f)-2: counting needs no line copies and no Python frame per batch of 16 results
        counted = _count_matches(file, patterns, [pattern_flags] * len(patterns), max_match_count, invert_match, fixed_strings)
        if counted is not None:
            return counted
    code = scan(
        file,
        patterns,
        _on_batch,
        flags=[pattern_flags] * len(patterns),
        max_match_count=max_match_count,
        buffer_count=_GREP_BATCH,
        invert_match=invert_match,
        before_context=before_context if context else 0,
        after_context=after_context if context else 0,
        fixed_strings=fixed_strings,
    )
    if only_matching:
        _fill_spans(groups, deferred, patterns, widths, python_patterns, errors, span_lines)
        collected = [entry for group in groups for entry in group]
    return (counter[0] if count_only else collected), code


class _MatchEnd(ctypes.Structure):
    """gpugrep_match_end (include/gpugrep.h)."""

    _fields_ = [("line_number", ctypes.c_ulonglong), ("id", ctypes.c_uint), ("end", ctypes.c_uint)]


def _span_widths(patterns: Sequence[str]) -> list[int] | None:
    """Fixed match width per pattern (-1: use re.finditer), or None if the loaded library cannot report match ends
    (a plain libhyperscanner.so)."""
    lib = _get_hyperscanner_lib()
    try:
        width = lib.gpugrep_span_width
        lib.gpugrep_match_ends  # pylint: disable=pointless-statement
    except AttributeError:
        return None
    width.restype = ctypes.c_int
    width.argtypes = [ctypes.c_char_p]
    return [width(pattern.encode()) for pattern in patterns]


class _MatchSpan(ctypes.Structure):
    """gpugrep_match_span (include/gpugrep.h)."""

    _fields_ = [("line_number", ctypes.c_ulonglong), ("start", ctypes.c_uint), ("end", ctypes.c_uint)]


_SPAN_OVER_BUDGET = 0xFFFFFFFF


def _span_exact(patterns: Sequence[str]) -> list[bool] | None:
    """Per pattern: True if the engine's leftmost-first match spans equal re.finditer() (gpugrep_span_exact), or None if the
    loaded library cannot compute spans."""
    lib = _get_hyperscanner_lib()
    try:
        exact = lib.gpugrep_span_exact
        lib.gpugrep_match_spans  # pylint: disable=pointless-statement
    except AttributeError:
        return None
    exact.restype = ctypes.c_int
    exact.argtypes = [ctypes.c_char_p]
    return [exact(pattern.encode()) == 1 for pattern in patterns]


class _SpanLines:
    """The records of the span route, per pattern id: ASCII lines ending in '\\n' of variable-width patterns that pass
    gpugrep_span_exact.  Whole batches are taken without a Python step per record: ids, line numbers and line pointers are
    read as three strided slices of the batch, and one isascii() / newline count over the joined lines checks the batch."""

    def __init__(self, widths: list[int], exact: list[bool]):
        self.routed = [width <= 0 and bool(ok) for width, ok in zip(widths, exact)]
        self.lines: dict[int, list] = {}   # pattern id -> [joined chunks, line numbers, line bytes, (output list, first, count)]

    def __len__(self) -> int:
        return sum(len(entry[1]) for entry in self.lines.values())

    def add(self, pattern_id: int, numbers: list[int], raws: list[bytes], groups: list, blob: bytes | None = None) -> None:
        entry = self.lines.setdefault(pattern_id, [[], [], [], []])
        out: list = []
        groups.append(out)   # filled by fill() with the entries of these lines
        entry[3].append((out, len(entry[1]), len(numbers)))
        entry[0].append(blob if blob is not None else b"".join(raws))
        entry[1].extend(numbers)
        entry[2].extend(raws)

    def take_batch(self, matches, count: int, groups: list) -> bool:
        """Takes the whole batch if every record belongs to one routed pattern and every line is ASCII and ends in '\\n'."""
        if count <= 0 or not any(self.routed):
            return False
        base = ctypes.cast(matches, ctypes.c_void_p).value   # hyperscanner_result_t: id @0, line_number @8, line @16
        ids = (ctypes.c_uint * (6 * count)).from_address(base)[0::6]
        pattern_id = ids[0]
        if pattern_id >= len(self.routed) or not self.routed[pattern_id] or ids.count(pattern_id) != count:
            return False
        raws = (ctypes.c_char_p * (3 * count)).from_address(base)[2::3]
        blob = b"".join(raws)
        # (a delivered line holds at most one '\\n', its last byte)
        if not blob.isascii() or blob.count(b"\n") != count:
            return False
        self.add(pattern_id, (ctypes.c_ulonglong * (3 * count)).from_address(base)[1::3], raws, groups, blob)
        return True

    def fill(self, patterns: Sequence[str], python_patterns: list, errors: str) -> None:
        for pattern_id, (chunks, numbers, raws, segments) in self.lines.items():
            entries, first_line = _span_entries(b"".join(chunks), numbers, raws, patterns[pattern_id], python_patterns[pattern_id], errors)
            for out, first, count in segments:
                lo = bisect.bisect_left(first_line, first)
                out.extend(entries[lo:bisect.bisect_left(first_line, first + count, lo)])


def _span_entries(text: bytes, numbers: list[int], raws: list[bytes], pattern: str, python_pattern, errors: str):
    """The `-o` entries (line number, part + '\\n') of the lines joined in `text`, from one gpugrep_match_spans call, and the
    index of the line of each entry.  A failed call, or a line over the step budget, takes re.finditer()."""
    lib = _get_hyperscanner_lib()
    spans = None
    found = ctypes.c_size_t(0)
    entry = getattr(lib, "gpugrep_match_spans", None)
    if entry is not None:
        entry.restype = ctypes.c_int
        entry.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                          ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
        capacity = 2 * len(numbers) + 1024
        for _ in range(2):
            spans = (_MatchSpan * capacity)()
            code = entry(text, len(text), 0, pattern.encode(), 262140, spans, capacity, ctypes.byref(found), None)
            if code != 0:
                spans = None
                break
            if found.value <= capacity:
                break
            capacity, spans = found.value, None
    if spans is None:
        entries, first_line = [], []
        for line, raw in enumerate(raws):
            parts = [(numbers[line] + 1, f"{part.group()}\n") for part in python_pattern.finditer(raw.decode(errors=errors))]
            entries += parts
            first_line += [line] * len(parts)
        return entries, first_line
    # the records as 32-bit words (line_number low / high, start, end), read in one step
    total = found.value
    words = (ctypes.c_uint * (4 * total)).from_buffer(spans)[:] if total else []
    lines, starts, ends = words[0::4], words[2::4], words[3::4]
    offsets = list(itertools.accumulate(map(len, raws), initial=0))
    whole = text.decode("ascii")
    if _SPAN_OVER_BUDGET not in starts:
        return [(numbers[line] + 1, whole[offsets[line] + start:offsets[line] + end] + "\n")
                for line, start, end in zip(lines, starts, ends)], lines
    entries, first_line = [], []
    for line, start, end in zip(lines, starts, ends):
        if start == _SPAN_OVER_BUDGET:
            parts = [(numbers[line] + 1, f"{part.group()}\n") for part in python_pattern.finditer(raws[line].decode(errors=errors))]
            entries += parts
            first_line += [line] * len(parts)
        else:
            entries.append((numbers[line] + 1, whole[offsets[line] + start:offsets[line] + end] + "\n"))
            first_line.append(line)
    return entries, first_line


def _fill_spans(groups: list, deferred: list, patterns: Sequence[str], widths: list[int] | None, python_patterns: list,
                errors: str, span_lines: _SpanLines | None = None) -> None:
    """SURVEY.md section 8(f-4): the spans of the records that the engine's answers cover.  Patterns of one fixed width
    (`deferred`) take ONE scan of their lines that reports every match end (gpugrep_match_ends, patterns compiled without
    flags like the reference's re.compile(pattern)): a pattern of fixed width w matches [end - w, end), and finditer()'s
    left-to-right, non-overlapping choice is a greedy pass over the ends.  The other patterns that pass the span screen
    (`span_lines`) take one gpugrep_match_spans call per pattern id, which returns the finditer() spans themselves.  Any
    failure falls back to re.finditer() for the records concerned."""
    if span_lines is not None:
        span_lines.fill(patterns, python_patterns, errors)
    if deferred:
        _fill_from_ends(groups, deferred, patterns, widths, python_patterns, errors)


def _fill_from_ends(groups: list, deferred: list, patterns: Sequence[str], widths: list[int], python_patterns: list,
                    errors: str) -> None:
    """The spans of fixed-width records from their match ends (gpugrep_match_ends)."""
    lib = _get_hyperscanner_lib()
    entry = lib.gpugrep_match_ends
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                      ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
    text = b"".join(raw for _, _, raw in deferred)
    # (ids = pattern indices here: the reference indexes its compiled patterns with the id of the record)
    pattern_array, flags_array, ids_array = prepare_patterns(patterns, flags=[0] * len(patterns), ids=list(range(len(patterns))))
    capacity = 4 * len(deferred) + 1024
    found = ctypes.c_size_t(0)
    ends = None
    for _ in range(2):
        ends = (_MatchEnd * capacity)()
        code = entry(text, len(text), 0, pattern_array, flags_array, ids_array, len(pattern_array), 262140, ends, capacity,
                     ctypes.byref(found), None)
        if code != 0:
            ends = None
            break
        if found.value <= capacity:
            break
        capacity, ends = found.value, None
    per_line: dict[int, list[int]] = {}
    if ends is not None:
        wanted = [pattern_id for _, pattern_id, _ in deferred]
        for k in range(found.value):
            item = ends[k]
            if item.id == wanted[item.line_number]:
                per_line.setdefault(item.line_number, []).append(item.end)
    for line, (slot, pattern_id, raw) in enumerate(deferred):
        number = groups[slot][0][0]
        if ends is None:
            parts = [part.group() for part in python_patterns[pattern_id].finditer(raw.decode(errors=errors))]
        else:
            width, last, parts = widths[pattern_id], 0, []
            for end in per_line.get(line, ()):   # ascending
                if end - width >= last:
                    parts.append(raw[end - width:end].decode(errors=errors))
                    last = end
        groups[slot] = [(number, f"{part}\n") for part in parts]
