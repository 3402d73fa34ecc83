"""Host reference of the search with mismatches (include/sufr_b200.h, sufr_b200_index_approx), computed from the text
and the set of indexed positions alone, with no suffix array: a sliding-window Hamming count over every indexed
position, under rules (a)-(c) of the header, grouped by the distinct matched string w."""
from itertools import combinations, product
from typing import Dict, Iterable, List, Sequence, Tuple

import numpy as np


def separators(text: bytes, starts: Sequence[int]) -> set:
    """Z: the last byte of the text and the byte before every sequence start c > 0."""
    z = {text[-1]} if text else set()
    return z | {text[c - 1] for c in starts if 0 < c <= len(text)}


def match_len(m: int, cap: int) -> int:
    """m' = min(m, cap) (cap 0: none)."""
    return min(m, cap) if cap else m


def matches(text: bytes, indexed: Iterable[int], query: bytes, k: int, cap: int, starts: Sequence[int]
            ) -> List[Tuple[bytes, int, List[int]]]:
    """(w, mismatches, sorted positions) of every match, in byte order of w."""
    n = len(text)
    m = match_len(len(query), cap)
    if m == 0 or m > n:
        return []
    t = np.frombuffer(text, np.uint8)
    q = np.frombuffer(query[:m], np.uint8)
    pos = np.sort(np.asarray(indexed if isinstance(indexed, np.ndarray) else list(indexed), dtype=np.int64))
    pos = pos[pos + m <= n]
    zmask = np.zeros(256, bool)
    zmask[list(separators(text, starts))] = True
    mis = np.zeros(len(pos), np.int64)
    bad = np.zeros(len(pos), bool)
    for j in range(m):
        c = t[pos + j]
        d = c != q[j]
        mis += d
        bad |= d & zmask[c]
    sel = (mis <= k) & ~bad
    groups: Dict[bytes, Tuple[int, List[int]]] = {}
    for p, e in zip(pos[sel].tolist(), mis[sel].tolist()):
        groups.setdefault(text[p:p + m], (e, []))[1].append(p)
    return [(w, e, ps) for w, (e, ps) in sorted(groups.items())]


def brute_force(text: bytes, indexed: Iterable[int], query: bytes, k: int, cap: int, starts: Sequence[int]
                ) -> List[Tuple[bytes, int, List[int]]]:
    """The same set by enumerating every Hamming neighbour of q[0, m') over the text's bytes (no separator at a
    substituted position) and finding each one with bytes.find."""
    n = len(text)
    m = match_len(len(query), cap)
    if m == 0 or m > n:
        return []
    z = separators(text, starts)
    alphabet = sorted(set(text) - z)
    indexed = set(indexed)
    q = query[:m]
    out = []
    seen = set()
    for e in range(k + 1):
        for where in combinations(range(m), e):
            choices = [[b for b in alphabet if b != q[j]] for j in where]
            for subs in product(*choices):
                w = bytearray(q)
                for j, b in zip(where, subs):
                    w[j] = b
                w = bytes(w)
                if w in seen:
                    continue
                seen.add(w)
                ps, at = [], text.find(w)
                while at >= 0:
                    if at in indexed:
                        ps.append(at)
                    at = text.find(w, at + 1)
                if ps:
                    out.append((w, e, ps))
    return sorted(out)
