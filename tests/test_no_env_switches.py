"""CPU: the library and the package read no environment variable, so results, launch shapes and workspace sizes do not
depend on the environment a process inherits."""
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_PARENT = os.path.join(ROOT, "nightcore-to-flac-analyzer_b200")


def _sources(sub, exts):
    top = os.path.join(PKG_PARENT, sub)
    for dirpath, _, files in os.walk(top):
        for f in sorted(files):
            if f.endswith(exts):
                yield os.path.join(dirpath, f)


def _hits(sub, exts, needles):
    out = []
    for path in _sources(sub, exts):
        with open(path, encoding="utf-8") as fh:
            for n, line in enumerate(fh, 1):
                if any(s in line for s in needles):
                    out.append(f"{os.path.relpath(path, ROOT)}:{n}: {line.strip()}")
    return out


def test_no_environment_reads_in_library_or_package():
    assert list(_sources("csrc", (".cu", ".cuh"))) and list(_sources("nightcore_analyzer", (".py",)))
    hits = _hits("csrc", (".cu", ".cuh", ".h", ".c", ".cpp"), ("getenv",))
    hits += _hits("nightcore_analyzer", (".py",), ("environ", "getenv"))
    assert not hits, "\n".join(hits)
