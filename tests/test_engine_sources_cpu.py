"""CPU test: the engine reads no environment variable, and no kernel reads the SM clock.

INTEGRATION.md §4 promises that loading and calling the library depends on no environment variable (the library only sets
CUDA_DEVICE_MAX_CONNECTIONS when it is unset), so no source under csrc may call getenv. Cycle stamps inside a kernel are product
instructions on every launch; kernel and stage times come from CUDA events (JxlB200LastStageTimes, bench.py) instead."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pdn-jpegxl_b200", "csrc")


def _sources(exts):
    for root, _, files in os.walk(CSRC):
        for f in sorted(files):
            if f.endswith(exts):
                path = os.path.join(root, f)
                with open(path, encoding="utf-8") as fh:
                    yield os.path.relpath(path, CSRC), fh.read()


def _hits(pattern, exts):
    return [(rel, n + 1, line.strip()) for rel, text in _sources(exts) for n, line in enumerate(text.splitlines()) if re.search(pattern, line)]


def test_sources_exist():
    assert len(list(_sources((".cu",)))) >= 8


def test_no_source_reads_the_environment():
    assert _hits(r"getenv\s*\(", (".cu", ".cuh", ".h", ".cc", ".inc")) == []


def test_no_device_source_reads_the_clock():
    # clock() / clock64() and the PTX special registers behind them (%clock, %clock64, %clock_hi, %globaltimer*) in inline asm
    assert _hits(r"\bclock(64)?\s*\(|%clock|%globaltimer", (".cu", ".cuh", ".h", ".inc")) == []
