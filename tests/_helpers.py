"""Small checkers shared by the parity tests."""
import numpy as np


def edit_distance(a, b):
    """Levenshtein distance of two strings / byte strings (row-vectorised DP; fine for a few thousand symbols)."""
    a = np.frombuffer(a.encode() if isinstance(a, str) else bytes(a), dtype=np.uint8)
    b = np.frombuffer(b.encode() if isinstance(b, str) else bytes(b), dtype=np.uint8)
    if len(a) == 0 or len(b) == 0:
        return max(len(a), len(b))
    prev = np.arange(len(b) + 1, dtype=np.int64)
    ar = np.arange(len(b) + 1, dtype=np.int64)
    for i in range(1, len(a) + 1):
        sub = prev[:-1] + (b != a[i - 1])
        best = np.minimum(sub, prev[1:] + 1)          # substitution / deletion
        # insertions: cur[j] = min_k<=j (cand[k] + j - k)  ->  running minimum of (cand[k] - k), plus j
        cand = np.concatenate(([i], best))
        prev = np.minimum.accumulate(cand - ar) + ar
    return int(prev[-1])


def at_sample(full, gold, name):
    """`full` at the indices of its last axis that the fixture stores `name` at (`<name>_idx`, oracle/make_golden.py)."""
    return np.asarray(full)[..., gold[name + "_idx"]]


def identity(a, b):
    """1 - edit distance / length of the longer string."""
    n = max(len(a), len(b), 1)
    return 1.0 - edit_distance(a, b) / n
