"""Shared helpers for the test-suite: golden fixtures and int <-> limb conversion via the oracle."""
import json
import os

import numpy as np

from oracle import oracle as O
from oracle import pyref as P

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bn254_golden.json")


def golden():
    with open(GOLDEN) as f:
        return json.load(f)


def ival(s):
    return int(s, 16)


def ipt(p):
    return None if p is None else (int(p[0], 16), int(p[1], 16))


def fr_arr(ints):
    return O.fr_from_ints([x % P.R for x in ints]) if len(ints) else np.zeros((0, 4), dtype=np.uint64)


def g1_arr(pts):
    return np.stack([O.g1_affine_from_ints(p) for p in pts]) if len(pts) else np.zeros((0, 8), dtype=np.uint64)


def mem_available():
    """MemAvailable of /proc/meminfo in bytes (0 when it cannot be read)"""
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0
