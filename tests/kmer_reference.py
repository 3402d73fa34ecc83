"""Host reference of the k-mer calls (include/sufr_b200.h), computed from the text alone: it never looks at the suffix
or LCP array, so it is independent of the arrays the GPU calls read.

A k-mer occurrence is a position p of record [a, e) with p + k <= e - 1 (the k bytes lie inside the record and never
include its last byte); in a DNA index all k bytes are A, C, G or T.  Records follow index_extract: record i owns
[c_i, c_{i+1}), the last one [c_{R-1}, n), positions before c_0 belong to [0, c_0), no starts = one record [0, n)."""
from collections import Counter
from typing import Dict, List, Sequence

import numpy as np


def record_ends(n: int, starts: Sequence[int]) -> np.ndarray:
    """end[p] = the end e of the record holding p."""
    cuts = sorted({int(c) for c in starts if 0 < c < n}) + [n]
    end = np.empty(n, dtype=np.int64)
    lo = 0
    for c in cuts:
        end[lo:c] = c
        lo = c
    return end


def occurrences(text: bytes, k: int, starts: Sequence[int], is_dna: bool) -> np.ndarray:
    n = len(text)
    if n == 0 or k < 1:
        return np.zeros(0, dtype=np.int64)
    end = record_ends(n, starts)
    p = np.arange(n, dtype=np.int64)
    ok = p + k <= end - 1
    if is_dna:
        t = np.frombuffer(text, dtype=np.uint8)
        bad = ~np.isin(t, np.frombuffer(b"ACGT", dtype=np.uint8))
        # bad bytes in [p, p + k): prefix sums
        c = np.concatenate([[0], np.cumsum(bad)])
        hi = np.minimum(p + k, n)
        ok &= (c[hi] - c[p]) == 0
    return p[ok]


def counts(text: bytes, k: int, starts: Sequence[int], is_dna: bool) -> Dict[bytes, int]:
    return Counter(text[p:p + k] for p in occurrences(text, k, starts, is_dna).tolist())


def distinct(text: bytes, k: int, starts: Sequence[int], is_dna: bool):
    """The distinct k-mers in byte order (the rank order of their groups: every key is k whole bytes) with counts."""
    c = counts(text, k, starts, is_dna)
    keys = sorted(c)
    return keys, [c[x] for x in keys]


def spectrum(text: bytes, k: int, starts: Sequence[int], is_dna: bool, num_bins: int):
    c = counts(text, k, starts, is_dna)
    h = np.zeros(num_bins, dtype=np.uint64)
    for v in c.values():
        h[min(v, num_bins) - 1] += 1
    return h, len(c), sum(c.values()), max(c.values(), default=0)


def multiplicity(text: bytes, k: int, starts: Sequence[int], is_dna: bool) -> np.ndarray:
    c = counts(text, k, starts, is_dna)
    out = np.zeros(len(text), dtype=np.uint32)
    for p in occurrences(text, k, starts, is_dna).tolist():
        out[p] = min(c[text[p:p + k]], 0xFFFFFFFF)
    return out


def groups_from_arrays(sa: Sequence[int], lcp: Sequence[int], k: int, occ: set) -> List[tuple]:
    """(rank_begin, rank_end, count, text position of the first occurrence) of the groups of a suffix / LCP array: a
    group starts at rank 0 and at every rank with LCP < k; count = its ranks whose suffix is an occurrence."""
    out, b = [], 0
    s = len(sa)
    for r in range(1, s + 1):
        if r == s or lcp[r] < k:
            occ_r = [sa[x] for x in range(b, r) if sa[x] in occ]
            out.append((b, r, len(occ_r), occ_r[0] if occ_r else None))
            b = r
    return out
