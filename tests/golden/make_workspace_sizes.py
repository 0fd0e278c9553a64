"""Print the SIZES table of tests/test_workspace_layout.py: every ncfa_*_workspace_bytes value on a grid of shapes, as
the built libncfa.so returns it.  The size queries need no device (without one the spectral query assumes the B200's
148 SMs).

    python __graft_entry__.py && python tests/golden/make_workspace_sizes.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "nightcore-to-flac-analyzer_b200"))
from nightcore_analyzer._native import lib  # noqa: E402

N_SEG = (1, 7, 125, 65535)
SEG_LEN = (0, 1, 511, 2048, 441_000, 3_969_000, 79_380_000)
HOPS = (64, 512, 96)
WINDOWS = (2756, 344)            # the 8 s tempogram window at hop 64 and hop 512 (sr 22 050)
ENV_LEN = sorted({1 + n // hop for n in SEG_LEN for hop in HOPS})


def grid():
    for n in N_SEG:
        yield "spectral", (n,)
        for m in (1, 3, 4, 64):
            yield "xcorr", (n, m)
        for a, b, n_boot in ((35, 27, 2000), (7, 0, 2000)):
            yield "bootstrap", (n, a, b, n_boot)
        for ln in SEG_LEN:
            yield "trim", (n, ln)
            yield "tuning", (n, ln)
            yield "chroma", (n, ln)
            for hop in HOPS:
                yield "onset", (n, ln, hop)
        for env in ENV_LEN:
            for w in WINDOWS:
                yield "tempo", (n, env, w)
                yield "beat", (n, env, w)
    yield "align", (30, 2585, 1000)


def main():
    rows = {}
    for fam, args in grid():
        rows.setdefault(fam, []).append(f"{args}: {getattr(lib, f'ncfa_{fam}_workspace_bytes')(*args)}")
    print("SIZES = {")
    for fam, items in rows.items():
        print(f'    "{fam}": {{')
        line = "       "
        for it in items:
            if len(line) + len(it) + 2 > 120:
                print(line)
                line = "       "
            line += f" {it},"
        print(line)
        print("    },")
    print("}")


if __name__ == "__main__":
    main()
