"""Host reference of the match set of a query over a suffix array index (numpy; no GPU).  Test helper only.

For an index (transformed text ``t``, suffix array, LCP array, build cap or seed mask) and a query, the suffixes that
match are found by comparing exact bytes at every text position, without looking at the suffix array order:

* no seed mask: with ``m`` the effective cap (the build cap, the run-time cap, or the smaller of the two; 0 and None
  both mean none) and ``k = min(len(q), m)``, suffix ``p`` matches iff ``p + k <= n`` and ``t[p:p+k] == q[:k]``;
* seed mask, query no longer than the mask: with ``c`` the care offsets below ``len(q)`` (under a run-time cap ``m``
  only the first ``m`` of them), suffix ``p`` matches iff every ``p + c < n`` and ``t[p + c] == q[c]``.

The matching ranks must be contiguous in the suffix array; the full-array answer is ``(first, last + 1)`` or None.
The in-memory answer (the LCP-subsampled array, ``sufr_search.rs:119-136``) follows from it and the LCP array: the
sampled ranks are those with ``lcp < eff``; the range starts at the first sampled rank in it; with one sampled rank in
it the range ends at the next sampled rank, or at the number of suffixes when there is none; with more than one it
ends at the last sampled rank + 1.

A seed-mask query LONGER than the mask (without a run-time cap at or below the weight) has no such definition: the
search then compares the byte right after the mask (``full_offset``), which the index order does not sort by.  For
those queries only, :func:`transcribed_search` is a plain transcription of ``compare`` / ``search_first`` /
``search_last`` (``sufr_search.rs:179-350``, as ``sufr_b200/csrc/search.cuh`` cites them).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

_KEY = 8                  # bytes of the packed key every text position is sorted by
_CONFIRM_CELLS = 1 << 24  # bytes compared per chunk when candidates are checked beyond the key


def mask_positions(mask: str) -> List[int]:
    return [i for i, c in enumerate(mask) if c == "1"]


@dataclass
class Index:
    """What the reference needs of an index.  ``build_mql`` is 0 for an uncapped one; ``seed_mask`` None without."""
    text: bytes
    sa: np.ndarray
    lcp: np.ndarray
    build_mql: int = 0
    seed_mask: Optional[str] = None
    t: np.ndarray = field(init=False, repr=False)
    rank_of: np.ndarray = field(init=False, repr=False)
    _sorted: Optional[Tuple[np.ndarray, np.ndarray]] = field(default=None, init=False, repr=False)
    _cache: Dict[Tuple[int, bytes], Optional[Tuple[int, int]]] = field(default_factory=dict, init=False, repr=False)

    def __post_init__(self):
        self.t = np.frombuffer(self.text, dtype=np.uint8)
        self.sa = np.asarray(self.sa).astype(np.int64)
        self.lcp = np.asarray(self.lcp).astype(np.int64)
        assert len(self.sa) == len(self.lcp) <= len(self.text)
        self.rank_of = np.full(len(self.text), -1, dtype=np.int64)
        self.rank_of[self.sa] = np.arange(len(self.sa), dtype=np.int64)
        assert len(np.unique(self.sa)) == len(self.sa)

    @property
    def n(self) -> int:
        return len(self.text)

    @property
    def s(self) -> int:
        return len(self.sa)

    @property
    def care(self) -> List[int]:
        return mask_positions(self.seed_mask) if self.seed_mask else []

    @property
    def built(self) -> int:
        """The max_query_len the index was built with, as sufr_file.rs:521-528 defines it."""
        if self.seed_mask:
            return len(self.care)
        return self.build_mql or self.n

    def subsample_cap(self, run_mql: Optional[int], low_memory: bool) -> Optional[int]:
        """The cap of the LCP-subsampled array an in-memory search uses, or None when it searches the full array."""
        if low_memory:
            return None
        eff = min(run_mql, self.built) if run_mql else self.built
        return eff if eff != self.built else None

    def offsets(self, count: int) -> List[int]:
        """The first ``count`` compared offsets: 0, 1, 2, ... or, with a seed mask, the care offsets."""
        return self.care[:count] if self.seed_mask else list(range(count))

    def sorted_keys(self) -> Tuple[np.ndarray, np.ndarray]:
        """Every text position with the bytes at its first 8 compared offsets packed into a u64 key (bytes past the
        end of the text read as 0), sorted by that key: (keys, positions).  Independent of the suffix array."""
        if self._sorted is None:
            base = self.offsets(_KEY)
            pad = np.concatenate([self.t, np.zeros(base[-1] + 1 if base else 1, dtype=np.uint8)])
            key = np.zeros(self.n, dtype=np.uint64)
            for o in base:
                key = (key << np.uint64(8)) | pad[o:o + self.n].astype(np.uint64)
            key <<= np.uint64(8 * (_KEY - len(base)))
            order = np.argsort(key, kind="stable")
            self._sorted = (key[order], order)
        return self._sorted


def _pack(b: bytes) -> int:
    v = 0
    for x in b:
        v = (v << 8) | x
    return v


def match_positions(idx: Index, offs: List[int], want: bytes) -> np.ndarray:
    """The text positions p with every p + o < n and t[p + o] == want[j] for the j-th offset o of ``offs`` (a
    non-empty prefix of idx.offsets): a range of the positions sorted by their first 8 bytes, then exact bytes."""
    keys, order = idx.sorted_keys()
    j = min(len(offs), _KEY)
    shift = 8 * (_KEY - j)
    lo = _pack(want[:j]) << shift
    a = int(np.searchsorted(keys, np.uint64(lo), side="left"))
    b = int(np.searchsorted(keys, np.uint64(lo | ((1 << shift) - 1)), side="right"))
    pos = np.sort(order[a:b])
    pos = pos[pos + offs[-1] < idx.n]
    if len(offs) > _KEY and len(pos):
        o = np.asarray(offs[_KEY:], dtype=np.int64)
        w = np.frombuffer(want[_KEY:], dtype=np.uint8)
        step = max(1, _CONFIRM_CELLS // len(o))
        keep = [(idx.t[pos[i:i + step, None] + o[None, :]] == w[None, :]).all(axis=1) for i in range(0, len(pos), step)]
        pos = pos[np.concatenate(keep)]
    return pos


def effective_cap(build_mql: int, run_mql: Optional[int]) -> int:
    """The cap of a comparison without a seed mask: 0 = none."""
    b, r = build_mql or 0, run_mql or 0
    if b and r:
        return min(b, r)
    return b or r


def needs_transcription(idx: Index, q: bytes, run_mql: Optional[int]) -> bool:
    """A seed-mask query longer than the mask, without a run-time cap at or below the weight."""
    if not idx.seed_mask or len(q) <= len(idx.seed_mask):
        return False
    return not (run_mql and run_mql <= len(idx.care))


def _pattern(idx: Index, q: bytes, run_mql: Optional[int]) -> Tuple[List[int], bytes]:
    """The offsets compared for q, and q's bytes at them."""
    if idx.seed_mask:
        c = [o for o in idx.care if o < len(q)]
        if run_mql:
            c = c[:run_mql]
        return c, bytes(q[o] for o in c)
    m = effective_cap(idx.build_mql, run_mql)
    k = min(len(q), m) if m else len(q)
    return idx.offsets(k), q[:k]


def full_ranges(idx: Index, queries: Sequence[bytes], run_mql: Optional[int] = None) -> List[Optional[Tuple[int, int]]]:
    """Per query the half-open range of matching ranks in the full suffix array, or None."""
    out = []
    for q in queries:
        q = bytes(q)
        if needs_transcription(idx, q, run_mql):
            out.append(transcribed_search(idx, q, run_mql))
            continue
        offs, want = _pattern(idx, q, run_mql)
        key = (len(offs), want)
        if key not in idx._cache:
            if not offs:  # nothing compared: every suffix matches
                idx._cache[key] = (0, idx.s) if idx.s else None
            else:
                r = idx.rank_of[match_positions(idx, offs, want)]
                r = r[r >= 0]
                lo, hi = (int(r.min()), int(r.max())) if len(r) else (0, -1)
                assert hi - lo + 1 == len(r), f"the matches of {q[:40]!r} are not contiguous in the suffix array"
                idx._cache[key] = (lo, hi + 1) if len(r) else None
        out.append(idx._cache[key])
    return out


def in_memory_range(full: Optional[Tuple[int, int]], sampled: np.ndarray, s: int) -> Optional[Tuple[int, int]]:
    """The answer of a search over the LCP-subsampled array, mapped back through the sampled ranks (``sampled``, the
    ranks with lcp < eff, ascending) as sufr_search.rs:119-136 does, from the full-array range ``full`` over an index
    of ``s`` suffixes."""
    if full is None:
        return None
    lo, hi = full
    a, b = np.searchsorted(sampled, lo), np.searchsorted(sampled, hi)
    if a == b:
        return None
    start = int(sampled[a])
    if b - a == 1:
        return start, int(sampled[a + 1]) if a + 1 < len(sampled) else s
    return start, int(sampled[b - 1]) + 1


def expected(idx: Index, queries: Sequence[bytes], run_mql: Optional[int], low_memory: bool,
             full: Optional[List[Optional[Tuple[int, int]]]] = None) -> List[Optional[Tuple[int, int]]]:
    """What ``SufrIndex.search(queries, run_mql, low_memory)`` returns.  ``full`` may pass full_ranges already
    computed for the same run-time cap."""
    if full is None:
        full = full_ranges(idx, queries, run_mql)
    eff = idx.subsample_cap(run_mql, low_memory)
    if eff is None:
        return list(full)
    sampled = np.flatnonzero(idx.lcp < eff)
    return [in_memory_range(r, sampled, idx.s) for r in full]


# ---------------------------------------------------------------- transcription (seed-mask queries beyond the mask)
def _full_offset(care: List[int], mask_len: int, lcp: int) -> int:
    """util.rs:19-37"""
    if lcp == 0 or lcp > mask_len:
        return lcp
    offset = care[lcp - 1]
    nxt = care[lcp] if lcp < len(care) else 0
    if nxt > offset and nxt - offset > 1:
        return nxt
    return offset + 1


def _compare(idx: Index, q: bytes, p: int, skip: int, run_mql: Optional[int]) -> Tuple[int, int]:
    """sufr_search.rs:261-350, seed-mask form: (lcp in care units, query vs suffix as -1 / 0 / 1)."""
    care, n, t = idx.care, idx.n, idx.text
    weight, mql = len(care), (run_mql or 0)
    if skip >= weight or (mql > 0 and skip >= mql):
        lcp = skip
    else:
        end = min(mql, weight) if mql > 0 else weight
        qn = sum(1 for k in range(skip, end) if care[k] < len(q))
        sn = sum(1 for k in range(skip, end) if p + care[k] < n)
        c = 0
        while c < min(qn, sn):
            off = care[skip + c]
            if p + off >= n or q[off] != t[p + off]:
                break
            c += 1
        lcp = skip + c
    if mql > 0 and lcp >= mql:
        return lcp, 0
    fo = _full_offset(care, len(idx.seed_mask), lcp)
    if fo >= len(q):
        return lcp, 0
    if p + fo >= n:
        return lcp, 1
    return lcp, (-1 if q[fo] < t[p + fo] else (1 if q[fo] > t[p + fo] else 0))


def transcribed_search(idx: Index, q: bytes, run_mql: Optional[int]) -> Optional[Tuple[int, int]]:
    """sufr_search.rs:179-249 over the full suffix array: (first, last + 1), or None."""
    sa = idx.sa
    ln = len(sa)
    low, high, left, right = 0, ln - 1, 0, 0
    first = -1
    while high >= low:
        mid = low + (high - low) // 2
        lcp, cmp = _compare(idx, q, int(sa[mid]), min(left, right), run_mql)
        if cmp == 0 and (mid == 0 or _compare(idx, q, int(sa[mid - 1]), 0, run_mql)[1] == 1):
            first = mid
            break
        if cmp == 1:
            low, left = mid + 1, lcp
        else:
            high, right = mid - 1, lcp
    if first < 0:
        return None
    low, high, left, right = first, ln - 1, 0, 0
    last = -1
    while high >= low:
        mid = low + (high - low) // 2
        lcp, cmp = _compare(idx, q, int(sa[mid]), min(left, right), run_mql)
        if cmp == 0 and (mid == ln - 1 or _compare(idx, q, int(sa[mid + 1]), 0, run_mql)[1] == -1):
            last = mid
            break
        if cmp == -1:
            high, right = mid - 1, lcp
        else:
            low, left = mid + 1, lcp
    if last < 0:
        last = first
    return first, last + 1
