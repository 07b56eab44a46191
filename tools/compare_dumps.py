"""Compares two `bench.py --dump-outputs` directories array by array.

    python tools/compare_dumps.py DIR_A DIR_B

Prints one JSON object: for every array, max |a - b| / max |a| (0.0 when bit-identical; null when the array is missing
on one side or the shapes differ)."""
import json
import os
import sys

import numpy as np


def compare(dir_a, dir_b):
    out = {}
    for name in sorted(set(os.listdir(dir_a)) | set(os.listdir(dir_b))):
        pa, pb = os.path.join(dir_a, name), os.path.join(dir_b, name)
        if not (os.path.exists(pa) and os.path.exists(pb)):
            out[name] = None
            continue
        a, b = np.load(pa).astype(np.float64), np.load(pb).astype(np.float64)
        out[name] = None if a.shape != b.shape else float(np.abs(a - b).max() / max(np.abs(a).max(), 1e-30))
    return out


if __name__ == "__main__":
    print(json.dumps(compare(sys.argv[1], sys.argv[2])))
