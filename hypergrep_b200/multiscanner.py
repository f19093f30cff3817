#! /usr/bin/env python3

"""grep-style command line over the GPU scan engine.

Mirror of the reference CLI (reference hypergrep/multiscanner.py): same options, same BRE/GNU pattern rewrites,
same output formats and exit codes (0 match, 1 no match, 2 error, 130 interrupted), one ``grep`` job per file.
Files are spread over the visible GPUs by the native library (one device per ``hyperscan`` call, round-robin),
which replaces the reference's "one CPU thread per file" scaling.
"""

from __future__ import annotations

import argparse
import multiprocessing
import re
import sys
import textwrap
from multiprocessing.pool import ThreadPool
from typing import Any, Iterable, Iterator

import hypergrep_b200 as hypergrep

_UNSUPPORTED_URL = "https://intel.github.io/hyperscan/dev-reference/compilation.html#unsupported-constructs"
# Characters that are literals in POSIX basic regular expressions unless escaped (and operators when escaped).
_BRE_SWAPPED = "+?(){}|"


def _grep_with_index(index: int, args: Iterable, kwargs: dict[str, Any]) -> tuple[int, Any]:
    """Pool job: run one grep and tag the outcome (result or exception) with its position in the file list."""
    try:
        outcome = hypergrep.grep(*args, **kwargs)
    except Exception as error:  # pylint: disable=broad-except
        outcome = error
    return index, outcome


def get_argparse_files(args: argparse.Namespace) -> list[str]:
    """Files named on the command line (reference multiscanner.py:27-43).

    As with GNU grep, once -e/-f supplied a pattern the bare positional "pattern" is really the first file.
    """
    files: list[str] = []
    if args.pattern and (args.patterns or args.pattern_files):
        files.append(args.pattern)
    files.extend(args.files or [])
    return files


def _validate_python_regex(pattern: str) -> None:
    try:
        re.compile(pattern)
    except Exception as error:
        raise ValueError(f"hyperscanner: invalid regex: {error}") from error


def get_argparse_patterns(args: argparse.Namespace) -> list[str]:
    """Patterns from the positional, -e and -f options, validated (reference multiscanner.py:46-83).

    Raises ValueError for patterns Python's ``re`` rejects and for patterns the engine's compiler rejects.
    """
    patterns: list[str] = []
    if args.patterns:
        patterns += args.patterns
    elif args.pattern and not args.pattern_files:
        patterns.append(args.pattern)
    for name in args.pattern_files or []:
        with open(name, "rt", encoding="utf-8") as handle:
            patterns += [line.rstrip("\n") for line in handle.readlines()]
    fixed = getattr(args, "regexp", None) == "fixed"
    if not fixed:   # (-F: literals, whatever Python's re thinks of them)
        for pattern in patterns:
            _validate_python_regex(pattern)
    # The compile check runs in the parent, before any pool exists, and never touches CUDA (fork-safe).
    if fixed and hypergrep.check_compatibility(patterns, fixed_strings=True):
        raise ValueError("hyperscanner: invalid fixed string")
    if not fixed and hypergrep.check_compatibility(patterns):
        raise ValueError(f"hyperscanner: incompatible regex: for more information visit {_UNSUPPORTED_URL}")
    return patterns


class _OrderedPrinter:  # pylint: disable=too-many-instance-attributes
    """Collects per-file outcomes from the pool and prints them, in file order unless told otherwise."""

    def __init__(self, files: list, options: dict[str, Any]) -> None:
        self.files = files
        self.opt = options
        self.waiting: dict[int, Any] = {}
        self.cursor = 0
        self.total = 0
        self.matched = False
        self.errored = False
        self.printed = False   # some line has been printed (a group separator goes before the next group)

    def __call__(self, tagged: tuple[int, Any]) -> None:
        index, outcome = tagged
        if self.opt["ordered_results"] and index != self.cursor:
            self.waiting[index] = outcome
            return
        self._report(index, outcome)

    def _advance(self) -> None:
        self.cursor += 1
        if self.cursor in self.waiting:
            self(((self.cursor), self.waiting.pop(self.cursor)))

    def _report(self, index: int, outcome: Any) -> None:
        name = self.files[index]
        if isinstance(outcome, Exception):
            print(f"hyperscanner: {name}: {outcome}")
            self.errored = True
            self._advance()
            return
        found, code = outcome
        if code:
            self.errored = True
        if found:
            self.matched = True
            if self.opt["quiet"]:
                return
        opt = self.opt
        if opt["files_without_match"]:
            if not found:
                print(name)
        elif opt["files_with_matches"]:
            if found:
                print(name)
        elif opt["total_results"]:
            self.total += found
        elif opt["count_results"]:
            print(f"{name}:{found}" if opt["with_file_name"] else f"{found}")
        else:
            try:
                if opt["context"]:
                    self.printed = print_context_results(found, name, opt["with_file_name"], opt["with_line_number"], opt["group_separator"],
                                                         opt["group_span"], self.printed)
                else:
                    print_results(found, name, with_file_name=opt["with_file_name"], with_line_number=opt["with_line_number"])
            except BrokenPipeError:
                pass  # e.g. piped into `head`; keep draining the pool
        self._advance()


def parallel_grep(  # pylint: disable=too-many-arguments,too-many-locals
    files: list,
    patterns: list[str],
    ignore_case: bool = False,
    ordered_results: bool = True,
    count_results: bool = False,
    total_results: bool = False,
    with_file_name: bool = False,
    with_line_number: bool = False,
    use_multithreading: bool = True,
    only_matching: bool = False,
    no_messages: bool = False,
    max_match_count: int = 0,
    files_without_match: bool = False,
    files_with_matches: bool = False,
    quiet: bool = False,
    invert_match: bool = False,
    before_context: int | None = None,
    after_context: int | None = None,
    group_separator: str | None = "--",
    fixed_strings: bool = False,
    word_regexp: bool = False,
    line_regexp: bool = False,
) -> int:
    """Scan files and print grep-formatted results (reference multiscanner.py:86-223).

    Returns the grep exit code: 2 if any file errored, else 1 if nothing matched, else 0.
    ``invert_match`` (``-v``) selects the lines that no pattern matches; every other option then applies to those lines.
    ``before_context`` / ``after_context`` (``-B`` / ``-A``) print the lines around each selected line, as GNU grep does,
    with ``group_separator`` (None: none) before each group that does not continue the previous output; as in GNU grep, a
    width of 0 still separates the groups, and None (the default) prints no context output at all.  -c, -t, -l, -L and
    -q ignore them; with -o only the matched parts are printed, and a separator goes between two selected lines whose gap
    exceeds ``before_context + after_context`` lines.
    ``fixed_strings`` (``-F``): the patterns are literals.
    ``word_regexp`` / ``line_regexp`` (``-F -w`` / ``-F -x``): a literal must occur as a whole word, or be the whole line;
    they need ``fixed_strings`` and do not combine with ``only_matching`` (ValueError).
    """
    if (word_regexp or line_regexp) and (only_matching or not fixed_strings):
        raise ValueError("word_regexp / line_regexp need fixed_strings and do not combine with only_matching")
    if invert_match and only_matching:
        # GNU grep -v -o: a selected line has no matching part, so nothing is printed; the exit code still says whether
        # some line was selected.  -c / -t / -l / -L keep their output.
        only_matching = False
        if not (count_results or total_results or files_with_matches or files_without_match):
            quiet = True
    if files_without_match or files_with_matches or quiet:
        max_match_count = 1  # these modes only need to know whether a file matches at all
    context = before_context is not None or after_context is not None
    if count_results or total_results or files_without_match or files_with_matches or quiet:
        context = False
    before_context, after_context = (before_context or 0, after_context or 0) if context else (0, 0)
    printer = _OrderedPrinter(
        files,
        {
            "ordered_results": ordered_results,
            "count_results": count_results,
            "total_results": total_results,
            "with_file_name": with_file_name,
            "with_line_number": with_line_number,
            "files_without_match": files_without_match,
            "files_with_matches": files_with_matches,
            "quiet": quiet,
            "context": context,
            "group_separator": group_separator,
            # printed lines continue a group when they are adjacent; with -o, selected lines whose windows touch
            "group_span": before_context + after_context + 1 if only_matching else 1,
        },
    )
    grep_kwargs = {
        "ignore_case": ignore_case,
        "count_only": count_results or total_results,
        "only_matching": only_matching,
        "no_messages": no_messages,
        "max_match_count": max_match_count,
        "invert_match": invert_match,
        # (-o prints matched parts only: the grouping of the selected lines is all the printer needs)
        "before_context": 0 if only_matching else before_context,
        "after_context": 0 if only_matching else after_context,
        "fixed_strings": fixed_strings,
        "word_regexp": word_regexp,
        "line_regexp": line_regexp,
    }
    workers = min(max(multiprocessing.cpu_count() - 1, 1), len(files))
    pool_type = ThreadPool if use_multithreading else multiprocessing.Pool
    with pool_type(processes=workers) as pool:
        pending = [
            pool.apply_async(_grep_with_index, (index, (name, patterns), grep_kwargs), callback=printer)
            for index, name in enumerate(files)
        ]
        for job in pending:
            job.get()
            if quiet and printer.matched:
                pool.terminate()
                break
    if total_results:
        print(printer.total)
    if printer.errored:
        return 2
    return 0 if printer.matched else 1


def print_results(results: list, file_name: str, with_file_name: bool = False, with_line_number: bool = False) -> None:
    """Print matched lines with the requested prefixes (reference multiscanner.py:226-255)."""
    prefix = f"{file_name}:" if with_file_name else ""
    if with_line_number:
        sys.stdout.write("".join(f"{prefix}{number}:{text}" for number, text in results))
    else:
        sys.stdout.write("".join(f"{prefix}{text}" for _, text in results))


def print_context_results(  # pylint: disable=too-many-arguments
    results: list, file_name: str, with_file_name: bool, with_line_number: bool, separator: str | None, span: int, printed: bool
) -> bool:
    """Print the results of a scan with context lines as GNU grep does: selected lines as ``name:12:text``, context lines as
    ``name-12-text``, and ``separator`` before each group that does not continue the previous output (``printed``: some
    line has been printed before, by any file).  A result continues the group when its line number is at most ``span``
    after the previous one.  ``results``: ``(number, text, is_context)``, or ``(number, part)`` with -o.  Returns ``printed``."""
    out = []
    previous = None
    for entry in results:
        number, text = entry[0], entry[1]
        mark = "-" if len(entry) > 2 and entry[2] else ":"
        if (previous is None or number - previous > span) and printed and separator is not None:
            out.append(f"{separator}\n")
        previous, printed = number, True
        out.append((f"{file_name}{mark}" if with_file_name else "") + (f"{number}{mark}" if with_line_number else "") + text)
    sys.stdout.write("".join(out))
    return printed


def read_stdin() -> Iterator[str]:
    """File names piped on stdin, one per line, until the first blank line or EOF."""
    for raw in iter(sys.stdin.readline, ""):
        name = raw.strip()
        if not name:
            return
        yield name


def to_basic_regular_expressions(patterns: list[str]) -> list[str]:
    """Rewrite PCRE/ERE syntax into what the same text means as a POSIX BRE (reference multiscanner.py:273-305).

    In a BRE the characters ``+?(){}|`` are literals and their escaped forms are the operators, so escaped and
    unescaped occurrences trade places.  Raises ValueError if the rewritten pattern is not a valid regex.
    """
    converted = []
    for pattern in patterns:
        out: list[str] = []
        for char in pattern:
            if char in _BRE_SWAPPED:
                if out and out[-1] == "\\":
                    out[-1] = char  # escaped in the input: becomes the bare operator
                else:
                    out.append("\\" + char)  # bare in the input: a literal in BRE
            else:
                out.append(char)
        rewritten = "".join(out)
        _validate_python_regex(rewritten)
        converted.append(rewritten)
    return converted


def to_gnu_regular_expressions(patterns: list[str]) -> list[str]:
    r"""Translate GNU word-edge escapes ``\<`` and ``\>`` to ``\b`` (reference multiscanner.py:308-328)."""
    return [re.sub(r"(?<!\\)\\[<>]", lambda _match: r"\b", pattern) for pattern in patterns]


_DESCRIPTION = """\
GPU grep (Global Regular Expression Print) for large log files.

Multi-pattern regex matching on NVIDIA B200 GPUs behind a grep-compatible command line:
    1. All patterns are compiled into one automaton set and matched in a single pass over the file.
    2. Files are read and decompressed (gzip, zstd) on host threads and scanned on the GPU.
    3. Several files are processed concurrently and spread over all visible GPUs.

Differences from standard "grep":
    1. Only the options listed here are supported.
    2. Patterns must avoid constructs that need backtracking (look-around, back-references, ...).
       More details: """ + _UNSUPPORTED_URL + """

Examples:
    hyperscanner <regex> <file(s)>
    find <args> | hyperscanner <regex>"""


def parse_args(args: list | None = None) -> argparse.Namespace:
    """Parse the command line; option names and destinations follow the reference (multiscanner.py:331-548)."""
    parser = argparse.ArgumentParser(
        formatter_class=argparse.RawTextHelpFormatter, add_help=False, description=textwrap.dedent(_DESCRIPTION)
    )
    parser.add_argument("pattern", nargs="?", help="Regex pattern to use.")
    parser.add_argument("files", nargs="*", help="Files to scan.")

    generic = parser.add_argument_group("Generic Program Information")
    generic.add_argument("--help", action="help", default=argparse.SUPPRESS, help="show this help message and exit")

    syntax = parser.add_argument_group("Pattern Syntax").add_mutually_exclusive_group()
    syntax.set_defaults(regexp="bre")
    for short, long_name, value, text in (
        ("-E", "--extended-regexp", "ere", "Interpret PATTERNS as extended regular expressions (EREs)."),
        ("-F", "--fixed-strings", "fixed", "Interpret PATTERNS as fixed strings, not regular expressions. Unlike GNU grep,\n"
                                           "an empty pattern is an error here (GNU grep matches every line)."),
        ("-G", "--basic-regexp", "bre", "Interpret PATTERNS as basic regular expressions. This is the default."),
        ("-P", "--perl-regexp", "pcre", "Interpret PATTERNS as Perl-compatible regular expressions (PCREs)."),
    ):
        syntax.add_argument(short, long_name, dest="regexp", action="store_const", const=value, help=text)

    matching = parser.add_argument_group("Matching Control")
    matching.add_argument("-e", "--regexp", action="append", dest="patterns", metavar="pattern",
                          help="Use PATTERNS as the patterns; may be repeated and combined with -f.")
    matching.add_argument("-f", "--file", action="append", dest="pattern_files", metavar="file",
                          help="Obtain patterns from FILE, one per line; may be repeated and combined with -e.")
    matching.add_argument("-i", "--ignore-case", action="store_true", help="Perform case insensitive matching.")
    matching.add_argument("-v", "--invert-match", action="store_true",
                          help="Invert the sense of matching, to select non-matching lines.")
    matching.add_argument("-w", "--word-regexp", action="store_true",
                          help="Select only lines in which a pattern occurs as a whole word: no [0-9A-Za-z_] byte\n"
                               "right before or after it. Needs -F here; does not combine with -o.")
    matching.add_argument("-x", "--line-regexp", action="store_true",
                          help="Select only lines that a pattern matches exactly (the whole line). Needs -F here;\n"
                               "does not combine with -o.")

    output = parser.add_argument_group("General Output Control")
    output.add_argument("-c", "--count", action="store_true",
                        help="Suppress normal output; print a count of matching lines for each input file.")
    output.add_argument("-L", "--files-without-match", action="store_true",
                        help="Suppress normal output; print the name of each input file without a match.")
    output.add_argument("-l", "--files-with-matches", action="store_true",
                        help="Suppress normal output; print the name of each input file with a match.")
    output.add_argument("-m", "--max-count", type=int, default=0, help="Stop reading a file after NUM matching lines.")
    output.add_argument("-o", "--only-matching", action="store_true",
                        help="Print only the matched (non-empty) parts of a matching line, one per output line.")
    output.add_argument("-q", "--quiet", "--silent", action="store_true",
                        help="Quiet; write nothing to standard output. Exit with zero status on the first match.")
    output.add_argument("-s", "--no-messages", action="store_true",
                        help="Suppress error messages about nonexistent or unreadable files.")

    prefix = parser.add_argument_group("Output Line Prefix Control")
    name_mode = prefix.add_mutually_exclusive_group()
    name_mode.add_argument("-H", "--with-filename", action="store_true", default=None,
                           help="Print the file name for each match (default with more than one file).")
    name_mode.add_argument("-h", "--no-filename", action="store_true", default=None,
                           help="Suppress the file name prefix (default with a single file).")
    prefix.add_argument("-n", "--line-number", action="store_true",
                        help="Prefix each line of output with the 1-based line number within its input file.")

    selection = parser.add_argument_group("File and Directory Selection")
    selection.add_argument("-a", "--text", action="store_true",
                           help="Accepted for grep compatibility; files are always processed as bytes.")

    context = parser.add_argument_group("Context Line Control")
    context.add_argument("-A", "--after-context", type=int, metavar="NUM", default=None,
                         help="Print NUM lines of trailing context after matching lines.")
    context.add_argument("-B", "--before-context", type=int, metavar="NUM", default=None,
                         help="Print NUM lines of leading context before matching lines.")
    context.add_argument("-C", "--context", type=int, metavar="NUM", default=None,
                         help="Print NUM lines of output context (-A and -B take precedence).")
    context.add_argument("--group-separator", metavar="SEP", default="--",
                         help="Print SEP on a line between groups of context lines (default: --).")
    context.add_argument("--no-group-separator", dest="group_separator", action="store_const", const=None,
                         help="Do not print a separator between groups of context lines.")

    extra = parser.add_argument_group("Unique arguments to hyperscanner")
    extra.add_argument("-t", "--total", action="store_true",
                       help="Suppress normal output; print a count of matching lines across all input files.")
    extra.add_argument("--no-gnu", dest="gnu_regexp", action="store_false",
                       help="Disable GNU grep compatibility rewrites of BRE/ERE patterns (\\< and \\> become \\b).")
    extra.add_argument("--no-order", dest="ordered", action="store_false",
                       help="Print results as files finish instead of in file order.")
    extra.add_argument("--no-sort", dest="sort_files", action="store_false",
                       help="Keep the given file order instead of sorting.")
    extra.add_argument("--mp", action="store_false", dest="use_multithreading",
                       help="Use a multiprocessing pool instead of threads.")

    parser.set_defaults(parser=parser)
    return parser.parse_intermixed_args(args=args)


def _usage_exit(args: argparse.Namespace) -> None:
    args.parser.print_usage()
    raise SystemExit(2)


def main() -> None:
    """Entry point of the ``hyperscanner`` command (reference multiscanner.py:551-606)."""
    args = parse_args()
    try:
        patterns = get_argparse_patterns(args)
        if not patterns:
            _usage_exit(args)
        if args.regexp == "bre":
            patterns = to_basic_regular_expressions(patterns)
    except ValueError as error:
        print(error)
        raise SystemExit(2) from error
    if (args.word_regexp or args.line_regexp) and (args.regexp != "fixed" or args.only_matching):
        print("hyperscanner: -w / -x need -F and do not combine with -o")
        raise SystemExit(2)
    if args.gnu_regexp and args.regexp not in ("pcre", "fixed"):
        patterns = to_gnu_regular_expressions(patterns)
    after_context = args.after_context if args.after_context is not None else args.context
    before_context = args.before_context if args.before_context is not None else args.context
    if after_context is not None or before_context is not None:   # (one given: the other is 0)
        after_context, before_context = after_context or 0, before_context or 0
    for value in (args.after_context, args.before_context, args.context):
        if value is not None and value < 0:
            print(f"hyperscanner: {value}: invalid context length argument")
            raise SystemExit(2)

    files = get_argparse_files(args) or list(read_stdin())
    if args.sort_files:
        files = sorted(files)
    if not files:
        _usage_exit(args)

    if args.no_filename is not None:
        with_file_name = False
    elif args.with_filename is not None:
        with_file_name = True
    else:
        with_file_name = len(files) > 1

    raise SystemExit(
        parallel_grep(
            files=files,
            patterns=patterns,
            ignore_case=args.ignore_case,
            ordered_results=args.ordered,
            count_results=args.count,
            total_results=args.total,
            with_file_name=with_file_name,
            with_line_number=args.line_number,
            use_multithreading=args.use_multithreading,
            only_matching=args.only_matching,
            no_messages=args.no_messages,
            max_match_count=args.max_count,
            quiet=args.quiet,
            files_without_match=args.files_without_match,
            files_with_matches=args.files_with_matches,
            invert_match=args.invert_match,
            before_context=before_context,
            after_context=after_context,
            group_separator=args.group_separator,
            fixed_strings=args.regexp == "fixed",
            word_regexp=args.word_regexp,
            line_regexp=args.line_regexp,
        )
    )


if __name__ == "__main__":
    try:
        main()
    except KeyboardInterrupt as interrupt:
        raise SystemExit(130) from interrupt
