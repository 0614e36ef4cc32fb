"""Generate tests/golden/live_golden.json: score and alignment digest (golden_io.results_digest) of every window of
golden_io.live_runs, the inputs on which tests compare with the unmodified reference, so that those tests check a fixed
result even where the reference is not built.  The results come from the unmodified reference (oracle/_ref/libclref.so)
where it is built, else from the C oracle, which reproduces every committed reference fixture; the file records which.
    python tests/golden/make_live_golden.py
"""
import json
import os
import sys

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)
from checkers import CpuChecker  # noqa: E402
from golden_io import LIVE_GOLDEN, live_runs, results_digest  # noqa: E402

NAMES = ("po_poa_oracle", "pwfa_oracle", "po_poa_gpu", "pwfa_gpu")


def main():
    kind = "reference" if CpuChecker.available("reference") else "port"
    chk = CpuChecker(kind)
    parts, n = [], 0
    for name in NAMES:  # one window per line
        runs = [results_digest(*chk.run(batch, p, lim)) for batch, p, lim in live_runs(name)]
        n += sum(len(r) for r in runs)
        parts.append(f'"{name}": [\n' + ",\n".join("[" + ",\n ".join(json.dumps(list(x)) for x in r) + "]" for r in runs) + "]")
    with open(LIVE_GOLDEN, "w") as f:
        f.write("{" + f'"checker": "{kind}",\n' + ",\n".join(parts) + "}\n")
    print(f"wrote {LIVE_GOLDEN} with the {kind} checker: {n} windows")


if __name__ == "__main__":
    main()
