"""Host reference of matching statistics and maximal exact matches (MEMs) over a suffix array index (numpy; no GPU).
Test helper only; the definitions are those of include/sufr_b200.h.

For a query ``q`` of length ``m`` and each ``0 <= i < m``, ``ms[i]`` is the largest ``l <= min(m - i, cap)`` such that
``q[i:i+l]`` is a prefix of some indexed suffix (a position the suffix array holds).  It is found by comparing the bytes
of every indexed suffix with the query's: the indexed positions are partitioned by their first one or two bytes, and
every position of the query's part is compared byte by byte, so the suffix array order plays no part.  The range ``[rb[i], re[i])`` is the set of ranks
of the suffixes left at the end, asserted to be contiguous; ``ms[i] = 0`` gives ``(NONE, NONE)``.

The MEMs with minimum length ``L`` are the ``(i, ms[i])`` with ``ms[i] >= L`` and (``i == 0`` or
``ms[i-1] <= ms[i]``), each with the occurrences ``SA[rb[i]:re[i]]``.  :func:`literal_mems` enumerates the maximal
exact matches of a query against a text pair by pair, from the definition alone, for the tests that pin the
maximality claim of an uncapped index.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Set, Tuple

import numpy as np

from search_reference import Index

NONE = 0xFFFFFFFFFFFFFFFF


class Matcher:
    """Matching statistics over ``idx`` with the build cap ``idx.build_mql`` (0 = none).  Seed-mask indexes have no
    matching statistics (include/sufr_b200.h) and are refused."""

    def __init__(self, idx: Index):
        assert not idx.seed_mask, "a seed-mask index has no matching statistics"
        self.idx = idx
        pos = np.sort(idx.sa)
        t = idx.t.astype(np.int64)
        # indexed positions by their first byte, and by their first two bytes: every indexed suffix that can share one
        # or two bytes with the query (a partition of all of them, not a use of their order)
        self._by_1: Dict[int, np.ndarray] = {}
        self._by_2: Dict[int, np.ndarray] = {}
        if len(pos):
            for b in np.unique(t[pos]):
                self._by_1[int(b)] = pos[t[pos] == b]
            two = pos[pos + 1 < idx.n]
            key = t[two] * 256 + t[two + 1]
            order = np.argsort(key, kind="stable")
            key, two = key[order], two[order]
            cuts = np.flatnonzero(np.diff(key)) + 1
            for k, grp in zip(np.split(key, cuts), np.split(two, cuts)):
                if len(k):
                    self._by_2[int(k[0])] = grp

    def _lcps(self, cand: np.ndarray, qa: np.ndarray, start: int, limit: int) -> np.ndarray:
        """Bytes q[i:i+limit] shares with the suffix at each candidate, given that all share the first `start`:
        compared in chunks that double, so long matches cost few passes."""
        t, n = self.idx.t, self.idx.n
        out = np.full(len(cand), start, dtype=np.int64)
        alive = np.arange(len(cand))
        off, w = start, 16
        while len(alive) and off < limit:
            w = min(w, limit - off)
            at = cand[alive, None] + off + np.arange(w)[None, :]
            eq = (at < n) & (t[np.minimum(at, n - 1)] == qa[off:off + w][None, :])
            run = np.where(eq.all(axis=1), w, np.argmin(eq, axis=1))
            out[alive] = off + run
            alive = alive[run == w]
            off, w = off + w, 2 * w
        return out

    def at(self, q: bytes, i: int) -> Tuple[int, int, int]:
        """(ms, rb, re) of position i of q."""
        idx = self.idx
        limit = len(q) - i
        if idx.build_mql:
            limit = min(limit, idx.build_mql)
        if limit <= 0 or q[i] not in self._by_1:
            return 0, NONE, NONE
        cand, start = self._by_1[q[i]], 1
        if limit >= 2 and q[i] * 256 + q[i + 1] in self._by_2:
            cand, start = self._by_2[q[i] * 256 + q[i + 1]], 2
        lcps = self._lcps(cand, np.frombuffer(q, np.uint8)[i:], start, limit)
        l = int(lcps.max())
        cand = cand[lcps == l]
        r = np.sort(idx.rank_of[cand])
        assert r[0] >= 0 and r[-1] - r[0] + 1 == len(r), \
            f"the suffixes starting with {q[i:i + l][:40]!r} are not contiguous in the suffix array"
        return l, int(r[0]), int(r[-1]) + 1

    def stats(self, q: bytes) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(ms, rb, re) of every position of q, numpy uint64."""
        rows = [self.at(q, i) for i in range(len(q))]
        cols = np.array(rows, dtype=np.uint64).reshape(len(q), 3)
        return cols[:, 0].copy(), cols[:, 1].copy(), cols[:, 2].copy()


def mems_of(ms: np.ndarray, rb: np.ndarray, re_: np.ndarray, min_len: int) -> List[Tuple[int, int, int, int]]:
    """The MEMs of one query from its matching statistics: (i, ms[i], rb[i], re[i])."""
    assert min_len >= 1
    out = []
    for i in range(len(ms)):
        if ms[i] >= min_len and (i == 0 or ms[i - 1] <= ms[i]):
            out.append((i, int(ms[i]), int(rb[i]), int(re_[i])))
    return out


def literal_mems(text: bytes, indexed: Set[int], q: bytes, min_len: int) -> Set[Tuple[int, int, int]]:
    """Every (i, p, l) with l >= min_len, p indexed, q[i:i+l] == text[p:p+l], that extends neither right
    (i + l == len(q), p + l == len(text) or the next bytes differ) nor left (i == 0, p == 0 or the bytes before differ),
    by comparing every pair of positions."""
    n, m = len(text), len(q)
    out = set()
    for i in range(m):
        for p in indexed:
            if i > 0 and p > 0 and q[i - 1] == text[p - 1]:
                continue
            l = 0
            while i + l < m and p + l < n and q[i + l] == text[p + l]:
                l += 1
            if l >= min_len:
                out.add((i, p, l))
    return out


def occurrences(idx: Index, mems: List[Tuple[int, int, int, int]]) -> Set[Tuple[int, int, int]]:
    """(i, SA[r], length) for every MEM and every rank r of its range."""
    return {(i, int(idx.sa[r]), l) for i, l, b, e in mems for r in range(b, e)}


def expected_stats(m: Matcher, queries: List[bytes]) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
    return [m.stats(bytes(q)) for q in queries]


def first_mismatch(got, want, queries) -> Optional[str]:
    """A readable description of the first position where two per-query (ms, rb, re) lists differ, or None."""
    for k, (g, w) in enumerate(zip(got, want)):
        for c, name in enumerate(("ms", "rank_begin", "rank_end")):
            a, b = np.asarray(g[c], np.uint64), np.asarray(w[c], np.uint64)
            head = f"query {k} ({bytes(queries[k])[:24]!r}, {len(queries[k])} bytes): {name}"
            if a.shape != b.shape:
                return f"{head} has {len(a)} entries, want {len(b)}"
            bad = np.flatnonzero(a != b)
            if len(bad):
                i = int(bad[0])
                return f"{head} differs at {len(bad)} positions, first i={i}: got {a[i]}, want {b[i]}"
    if len(got) != len(want):
        return f"{len(got)} queries answered, want {len(want)}"
    return None
