"""The C-ABI library loads without a GPU, exports every symbol include/gpugrep.h declares, and fails loudly (no CPU
fallback) when asked to scan without a CUDA device."""

import ast
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "gpugrep.h"), encoding="utf-8") as handle:
        text = handle.read()
    return sorted(set(re.findall(r"GPUGREP_API\s+[\w\s\*]+?\b(\w+)\(", text)))


def test_header_symbols_are_exported(gpu_lib):
    names = _declared_symbols()
    assert "hyperscan" in names and "check_patterns" in names and len(names) >= 16
    for name in names:
        assert hasattr(gpu_lib, name), f"{name} declared in include/gpugrep.h but not exported"


def test_synth_library_is_separate(gpu_lib):
    """The corpus generator lives in libgpugrep_synth.so (include/gpugrep_synth.h), not in the product library."""
    synth = ctypes.CDLL(os.path.join(ROOT, "hypergrep_b200", "lib", "libgpugrep_synth.so"))
    assert hasattr(synth, "gpugrep_synth_syslog") and not hasattr(gpu_lib, "gpugrep_synth_syslog")


def test_result_layout_matches_reference():
    from hypergrep_b200 import Result

    assert ctypes.sizeof(Result) == 24
    assert Result.id.offset == 0 and Result.line_number.offset == 8 and Result.line.offset == 16


def test_check_patterns_needs_no_gpu(gpu_lib):
    import hypergrep_b200 as hg

    assert hg.check_compatibility(["foobar"]) == 0
    assert hg.check_compatibility(["(?<!foo)bar"]) == 4          # reference test_hypergrep.py:64-74
    assert hg.check_compatibility(["a*"]) == 4                    # matches the empty buffer
    assert hg.check_compatibility(["foo"], flags=[64]) == 4       # unsupported flag bit
    with pytest.raises(ValueError):
        hg.check_compatibility([""])


def test_scan_without_gpu_fails_loudly(gpu_lib, tmp_path):
    """In a fresh interpreter that sees no CUDA device (CUDA_VISIBLE_DEVICES=""), also on a machine that has one."""
    path = tmp_path / "a.txt"
    path.write_text("foo\n")
    script = "import sys; import hypergrep_b200 as hg; print(hg.grep(sys.argv[1], ['foo']))"
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=ROOT)
    proc = subprocess.run([sys.executable, "-c", script, str(path)], env=env, capture_output=True, text=True, timeout=300, check=False)
    assert proc.returncode == 0, proc.stdout + proc.stderr
    results, code = ast.literal_eval(proc.stdout.strip())
    assert results == [] and code == 3   # HYPERSCANNER_SCRATCH: no device, and no CPU path to fall back to
