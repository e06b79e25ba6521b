"""The environment variables the library reads are exactly the ones DESIGN.md's tuning-knob table documents, and they are read
in one place (read_raycast_knobs in csrc/raycast_shadow.cu)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "isaac_rover_2.0_b200", "csrc")


def _sources():
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh")):
            with open(os.path.join(CSRC, f)) as fh:
                yield f, fh.read()


def _strip_comments(src):
    return re.sub(r"//[^\n]*|/\*.*?\*/", "", src, flags=re.S)


def test_knobs_read_by_the_library_are_the_documented_ones():
    read = set()
    for _, src in _sources():
        read |= set(re.findall(r'"(RVB_[A-Z0-9_]+)"', _strip_comments(src)))
    with open(os.path.join(ROOT, "DESIGN.md")) as fh:
        design = fh.read()
    section = design[design.index("### Tuning knobs"):]
    section = section[:section.index("\n## ")]
    table = [line for line in section.splitlines() if line.startswith("| `")]
    documented = {re.match(r"\| `(RVB_[A-Z0-9_]+)`", line).group(1) for line in table}
    assert read == documented
    assert len(read) == 6


def test_getenv_only_in_the_knob_reader():
    calls = [(f, src.count("getenv(")) for f, src in _sources() if "getenv(" in _strip_comments(src)]
    assert calls == [("raycast_shadow.cu", 1)]
