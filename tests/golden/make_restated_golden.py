#!/usr/bin/env python
"""Store the answers tests/test_restated_golden.py checks: what the workload generators, the oracle's leaf functions and
the host BVH builder return on the inputs of the live reference comparisons (tests/test_harness.py, test_oracle_units.py,
test_oracle_golden.py, test_builder.py). Regenerate only from a tree whose live comparisons pass against the reference's
own build (oracle/_ref), so that the stored answers are the reference's.   python tests/golden/make_restated_golden.py
Output: tests/golden/restated_golden.npz
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.pyoracle import Port  # noqa: E402
from tests.test_restated_golden import COMPUTE, GOLDEN  # noqa: E402


def main():
    port = Port()
    blob = {f"{group}/{k}": v for group, fn in COMPUTE.items() for k, v in fn(port).items()}
    np.savez_compressed(GOLDEN, **blob)
    print(f"wrote {GOLDEN}: {len(blob)} arrays, {os.path.getsize(GOLDEN) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
