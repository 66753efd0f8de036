"""Reference answers for batched exact-match queries (Context.locate / asgart_b200_ctx_locate): the oracle's sa_search
restatement (oracle.sa_search_literal, pinned to the reference's sa_searchb64 in tests/test_oracle_ref.py) over a batch,
a brute force over sorted suffixes, and the pattern sets the tests use."""
from typing import List, Sequence, Tuple

import numpy as np

import oracle

FOREIGN = [b"N", b"$", b"a", b"c", b"n", b"\x00", b"\xff", b"B", b"Z", b"-"]


def sa_search_batch(text, patterns: Sequence[bytes], sa: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """oracle.sa_search_literal for every pattern: (first int64[n], count int64[n])."""
    t = oracle.as_strand(text)
    sa = np.ascontiguousarray(sa, dtype=np.int64)
    out = [oracle.sa_search_literal(t, p, sa) for p in patterns]
    return (np.array([o[0] for o in out], dtype=np.int64).reshape(-1), np.array([o[1] for o in out], dtype=np.int64).reshape(-1))


def sorted_suffixes(text) -> np.ndarray:
    """Suffix array by sorting the suffixes as bytes (a suffix that is a prefix of another sorts first)."""
    t = bytes(oracle.as_strand(text))
    return np.array(sorted(range(len(t)), key=lambda i: t[i:]), dtype=np.int64)


def brute_force(text, patterns: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """(first, count) over all suffixes, sorted: count = suffixes that start with P, first = suffixes smaller than P
    (compared over at most len(P) bytes; one that ends inside P is smaller)."""
    t = bytes(oracle.as_strand(text))
    sa = sorted_suffixes(t)
    first, count = [], []
    for p in patterns:
        heads = [t[i:i + len(p)] for i in sa]
        first.append(sum(h < p for h in heads))
        count.append(sum(h == p for h in heads))
    return np.array(first, dtype=np.int64), np.array(count, dtype=np.int64)


def patterns_for(strand: np.ndarray, seed: int, lengths: Sequence[int], per_length: int = 4, foreign: bool = True) -> List[bytes]:
    """Per length: half cut from the strand (hits; some near its end, so they run past the '$'), half random ACGT
    (misses at the longer lengths); then copies with a foreign byte (N, '$', lower case, 0x00, 0xFF, 'B', ...) put in."""
    rng = np.random.default_rng(seed)
    t = bytes(oracle.as_strand(strand))
    n1 = len(t)
    out: List[bytes] = []
    for L in lengths:
        for j in range(per_length):
            if j % 2 == 0:
                x = int(rng.integers(0, n1)) if j % 4 == 0 else max(0, n1 - 1 - int(rng.integers(0, max(1, min(L, n1)))))
                p = t[x:x + L]
                if len(p) < L:   # runs past the end of the strand
                    p += bytes(rng.choice(list(b"ACGT"), L - len(p)).astype(np.uint8))
            else:
                p = bytes(rng.choice(list(b"ACGT"), L).astype(np.uint8))
            out.append(p)
            if foreign and L > 0 and j < 2:
                f = FOREIGN[int(rng.integers(0, len(FOREIGN)))]
                at = int(rng.integers(0, L))
                out.append(p[:at] + f + p[at + 1:])
    out += [b"", b"$", b"A$", b"N" * 3, b"\x00", b"\xff", b"B", b"a", b"ACGT" * 10 + b"\x00"]
    return out
