"""CPU test: every kernel launch of the engine goes through Launch (csrc/dev/kernels.h).

Launch opts a kernel in to its dynamic shared memory, checks that the runtime accepted the launch and counts it for
JxlB200KernelLaunchCount. A launch written anywhere else would return Ok when the runtime refuses it, so the triple-chevron syntax
and the shared-memory attribute call may appear only inside Launch and AllowDynamicSmem, and the old manual counter is gone."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pdn-jpegxl_b200", "csrc")
HELPER = os.path.join("dev", "kernels.h")


def _sources():
    for root, _, files in os.walk(CSRC):
        for f in sorted(files):
            if f.endswith((".cu", ".cuh", ".h", ".cc", ".inc")):
                path = os.path.join(root, f)
                with open(path, encoding="utf-8") as fh:
                    yield os.path.relpath(path, CSRC), fh.read()


def _hits(pattern):
    return [(rel, n + 1, line.strip()) for rel, text in _sources() for n, line in enumerate(text.splitlines()) if re.search(pattern, line)]


def _body(name):
    """Source of the helper function `name`, from its declaration to the closing brace at column 0."""
    with open(os.path.join(CSRC, HELPER), encoding="utf-8") as fh:
        text = fh.read()
    m = re.search(r"\b" + name + r"\(", text)
    assert m, name + " not found in " + HELPER
    return text[m.start():text.index("\n}\n", m.start())]


def test_kernels_are_launched_only_by_the_helper():
    hits = _hits(r"<<<")
    assert [(rel, line) for rel, _, line in hits] == [(HELPER, "Kernel<<<grid, block, smem, st>>>(args...);")], hits
    assert "<<<" in _body("Launch")


def test_shared_memory_attribute_is_set_only_by_the_helper():
    hits = _hits(r"\bcudaFuncSetAttribute\b")
    assert len(hits) == 1 and hits[0][0] == HELPER, hits
    assert "cudaFuncSetAttribute" in _body("AllowDynamicSmem")


def test_no_manual_launch_counting():
    assert _hits(r"\bCountLaunch\b") == []
