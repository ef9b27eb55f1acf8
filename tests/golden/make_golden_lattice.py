"""Generates tests/golden/lattice/*.npz, what tests/test_oracle.py::test_port_vs_reference_build compares the C
restatement with:

    python tests/golden/make_golden_lattice.py

For each (kind, shape) case of that test it stores, for every array of tests/test_oracle.py:lattice_case_arrays
(filtered tensors of both wrappers, offset_, barycentric_, neighbour table and M of the first frame's two lattices),
the SHA-256 of its bytes, its dtype, shape and float64 sum; the digests keep the files at about a kilobyte.  The
arrays come from the reference build (oracle/_ref) when it is present, else from the C restatement; `made_by` says
which.  The restatement matched the reference build bit for bit on exactly these cases (the same test, run against
oracle/_ref), and neither it nor the input generator has changed since, so both give the same bytes; wherever
oracle/_ref is built the test compares the restatement with it again.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

import oracle  # noqa: E402
from test_oracle import LATTICE_KINDS, LATTICE_SHAPES, lattice_case_arrays, lattice_case_name, sha256_of  # noqa: E402

OUT = os.path.join(HERE, "lattice")


def main():
    oracle.load_port()
    ref = oracle.have_ref()
    os.makedirs(OUT, exist_ok=True)
    for kind in LATTICE_KINDS:
        for shape in LATTICE_SHAPES:
            entries = {"made_by": "reference" if ref else "port"}
            for key, a in lattice_case_arrays(oracle, kind, shape, ref).items():
                entries[key + "_sha256"] = sha256_of(a)
                entries[key + "_dtype"] = str(a.dtype)
                entries[key + "_shape"] = np.array(a.shape, dtype=np.int64)
                entries[key + "_sum"] = np.float64(a.sum(dtype=np.float64))
            path = os.path.join(OUT, lattice_case_name(kind, shape) + ".npz")
            np.savez_compressed(path, **entries)
            print(path, os.path.getsize(path), "bytes, made by", entries["made_by"])


if __name__ == "__main__":
    main()
