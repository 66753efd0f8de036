"""Generate tests/golden/trim_search_golden.json: the reference's (first, count) for every pattern of
tests/test_oracle_ref.py::trim_cases, looked up in suffix arrays of trimmed strands (bin/asgart.rs:142-155). Near the cut
such an array is not sorted for the whole strand, so the answer is whatever the reference's bisection lands on: only
the reference's own steps give it, not a definition.

    python tests/golden/make_trim_golden.py

With oracle/_ref built, the answers come from the reference's sa_searchb64 over the whole array. Without it, they come
from `sa_search` below, a transcription of libdivsufsort's sa_search (lib/utils.c), written apart from the oracle's C++
restatement so that the two check each other. The file records which source was used.
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from tests.test_oracle_ref import TRIMS, trim_cases  # noqa: E402


def _compare(T: bytes, P: bytes, suf: int, match: int):
    """libdivsufsort's _compare: (< 0, 0, > 0 as suffix `suf` sorts before, starts with, or sorts after P; new match)."""
    i, j, r = suf + match, match, 0
    while i < len(T) and j < len(P):
        r = T[i] - P[j]
        if r != 0:
            break
        i, j = i + 1, j + 1
    else:
        r = 0
    return (-int(j != len(P)) if r == 0 else r), j


def sa_search(T: bytes, P: bytes, SA) -> tuple:
    """libdivsufsort's sa_search: (first index, count) of the suffixes that start with P, found by its bisection."""
    if len(T) == 0 or len(SA) == 0:
        return -1, 0
    if len(P) == 0:
        return 0, len(SA)
    i = j = k = 0
    lmatch = rmatch = 0
    size, half = len(SA), len(SA) >> 1
    while size > 0:
        r, match = _compare(T, P, SA[i + half], min(lmatch, rmatch))
        if r < 0:
            i += half + 1
            half -= (size & 1) ^ 1
            lmatch = match
        elif r > 0:
            rmatch = match
        else:
            lsize, j, rsize, k = half, i, size - half - 1, i + half + 1
            llmatch, lrmatch, half = lmatch, match, lsize >> 1
            while lsize > 0:                              # left part: first suffix that starts with P
                r, lmatch = _compare(T, P, SA[j + half], min(llmatch, lrmatch))
                if r < 0:
                    j += half + 1
                    half -= (lsize & 1) ^ 1
                    llmatch = lmatch
                else:
                    lrmatch = lmatch
                lsize, half = half, half >> 1
            rlmatch, rrmatch, half = match, rmatch, rsize >> 1
            while rsize > 0:                              # right part: one past the last
                r, rmatch = _compare(T, P, SA[k + half], min(rlmatch, rrmatch))
                if r <= 0:
                    k += half + 1
                    half -= (rsize & 1) ^ 1
                    rlmatch = rmatch
                else:
                    rrmatch = rmatch
                rsize, half = half, half >> 1
            break
        size, half = half, half >> 1
    return (j if k - j > 0 else i), k - j


def main():
    R = oracle.ref()
    t, trims = trim_cases()
    T = bytes(t)
    out = []
    for a, b, sa, pats in trims:
        first, count = [], []
        for p in pats:
            if R is not None:
                pa = np.frombuffer(p, dtype=np.uint8)
                idx = C.c_int64()
                c = R.sa_searchb64(t.ctypes.data, len(t), pa.ctypes.data, len(pa), sa.ctypes.data, len(sa), C.byref(idx), 0, len(sa))
                f = idx.value
            else:
                f, c = sa_search(T, p, sa.tolist())
            first.append(int(f))
            count.append(int(c))
        out.append({"a": a, "b": b, "first": first, "count": count})
    source = ("reference libdivsufsort sa_searchb64 (oracle/_ref)" if R is not None
              else "transcription of libdivsufsort lib/utils.c sa_search (tests/golden/make_trim_golden.py)")
    with open(os.path.join(os.path.dirname(__file__), TRIMS), "w") as f:
        json.dump({"generator": "tests/golden/make_trim_golden.py", "source": source,
                   "text_sha256": hashlib.sha256(t.tobytes()).hexdigest(), "trims": out}, f, separators=(",", ":"))
    print("wrote", sum(len(x["first"]) for x in out), "answers from", source)


if __name__ == "__main__":
    main()
