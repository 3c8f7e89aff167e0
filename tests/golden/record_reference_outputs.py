"""Writes tests/golden/reference_outputs.npz: what the reference's own compiled code (DUNE-DAQ fdreadoutlibs, its headers built
unmodified behind oracle/ref_wrapper.cpp) returns for every input of tests/test_oracle_vs_reference.py and of the GPU tests
that compare with the reference itself (the runs of tests/cases.py:reference_runs). With it those comparisons run without
the reference.

The outputs are recorded from the oracle (oracle/swtpg_oracle.c), and only from the exact source pinned below. At commit
6a0f75b, which has this oracle source, every one of those comparisons passed against the live reference library: 122 CPU
tests (the 52 of tests/test_oracle_vs_reference.py among them) and 139 GPU tests. On these inputs the oracle's outputs are
therefore the reference's outputs. Any other oracle source is refused, because its outputs are not known to be the
reference's.

    python tests/golden/record_reference_outputs.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import cases  # noqa: E402
from util import digest  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_outputs.npz")
MAX_STORED_BYTES = 8192
PINNED_ORACLE = {
    "oracle/swtpg_oracle.c": "e628a7ea5cffcf0ed14af27586a05f23ca82a1105b6ee5e3bf116d4964425105",
    "oracle/swtpg_oracle.h": "ce6f823fa8f5e0ca737bddc3e8dc9646c3967da4d18806a40c25db34797e127f",
}


def main():
    for path, want in PINNED_ORACLE.items():
        with open(os.path.join(ROOT, path), "rb") as f:
            if hashlib.sha256(f.read()).hexdigest() != want:
                sys.exit(f"{path} is not the oracle source that was checked against the reference; not recording")
    blobs = {}
    for key, run in cases.reference_runs():
        for name, a in run().items():
            k = f"{key}__{name}"
            if a.nbytes <= MAX_STORED_BYTES:
                blobs[k] = a
            else:  # kept small: the length and digest of a long array
                blobs[k + "_count"] = np.array([a.size], dtype=np.int64)
                blobs[k + "_sha256"] = digest(name, a)
    np.savez_compressed(OUT, **blobs)
    print(f"wrote {OUT}: {len(blobs)} arrays, {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
