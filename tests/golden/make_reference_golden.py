"""Writes tests/golden/reference_cases.npz: the outputs of the cases of tests/reference_cases.py.

The values come from the oracle. tests/test_reference_pwn_core.py requires the oracle to be bit-identical to the
reference's own pwn_core sources on each of these cases (omega and the eigen-ratios to rounding), so the file holds
what the reference computes. Where oracle/_ref/libpwn_core_ref.so is built, run that module before regenerating.

    python tests/golden/make_reference_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import reference_cases as RC  # noqa: E402
from test_reference_golden import GOLDEN, record  # noqa: E402


def main():
    rec = {}
    for case, fn in sorted(RC.all_cases().items()):
        rec.update(record(case, fn()))
    np.savez_compressed(GOLDEN, **rec)
    print("wrote %s: %d cases, %d bytes" % (GOLDEN, len(RC.all_cases()), os.path.getsize(GOLDEN)))


if __name__ == "__main__":
    main()
