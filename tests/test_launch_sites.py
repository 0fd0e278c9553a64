"""CPU: every kernel launch in csrc/ goes through ncfa::launch (ncfa_common.cuh), so each one is profiled under its
name, gets its dynamic shared-memory limit raised and has its launch error checked."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "nightcore-to-flac-analyzer_b200", "csrc")


def _code(path):
    """Source without comments, so prose may still mention ProfScope."""
    with open(path, encoding="utf-8") as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", lambda m: "\n" * m.group(0).count("\n"), text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def _block(text, start):
    """From the line that contains `start` to the first line that closes a top-level brace."""
    i = text.index(start)
    i = text.rindex("\n", 0, i) + 1
    return text[i : text.index("\n}", i) + 3]


def test_kernels_launch_only_through_the_helper():
    files = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))
    assert "ncfa_common.cuh" in files
    hits = []
    for f in files:
        text = _code(os.path.join(CSRC, f))
        if f == "ncfa_common.cuh":
            helper = _block(text, "int launch(")
            assert helper.count("<<<") == 1 and "ProfScope" in helper
            text = text.replace(helper, "").replace(_block(text, "struct ProfScope {"), "")
        for n, line in enumerate(text.splitlines(), 1):
            if "<<<" in line or "ProfScope" in line or "NCFA_LAUNCH_OK" in line:
                hits.append(f"{f}:{n}: {line.strip()}")
    assert not hits, "\n".join(hits)
