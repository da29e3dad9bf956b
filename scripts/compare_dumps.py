#!/usr/bin/env python
"""Compare two `bench.py --dump-outputs DIR` directories, e.g. of two builds run with the same arguments: the inputs are seeded, so
the same rows must come out.  Every array is compared exactly (the dumped values are integer counts and keys).  Exits with status 1
when a file is missing on one side or differs.

  python scripts/compare_dumps.py DIR_A DIR_B
"""
import os
import sys

import numpy as np


def main(argv):
    if len(argv) != 3:
        sys.exit(__doc__.strip().splitlines()[-1].strip())
    a, b = argv[1], argv[2]
    fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
    only = sorted(set(fa) ^ set(fb))
    bad = [f for f in sorted(set(fa) & set(fb)) if not np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f)))]
    print("dump files", len(set(fa) | set(fb)), "only on one side", only, "differing", bad)
    return 1 if only or bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
