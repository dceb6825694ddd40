"""Writes tests/golden/reference_outputs.json: a SHA-256 of every array tests/test_oracle_vs_reference.py compares, for
each of its seeded inputs, so that the test pins the C restatement without the reference's own classes at hand.

The arrays come from the reference's own decoder classes (oracle/_ref, built by `make -C oracle ref` from the upstream
Pheniqs sources) where they are built, else from the C restatement; the file records which under "source". A file
from the restatement pins it to what it computes today, which the live comparison found bit identical to the reference
wherever oracle/_ref was present.

Run from the repository root after build():  python tests/golden/make_reference_vectors.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import oracle as O  # noqa: E402
import test_oracle_vs_reference as V  # noqa: E402


def main():
    reference = O.ref_available()
    out = {"source": "reference (oracle/_ref)" if reference else "C restatement (oracle/libpheniqs_oracle.so)"}
    for key, inputs in V.cases():
        compiled, batch, n_segments = inputs()
        checker = O.RefOracle(compiled, n_segments) if reference else O.PortOracle(compiled)
        out[key] = V.digests(V.outputs(checker, batch))
    with open(os.path.join(ROOT, "tests", "golden", "reference_outputs.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
