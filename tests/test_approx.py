"""Search with mismatches on a device index (sufr_b200_index_approx / _approx_matches, SufrIndex.approx_matches /
.locate_approx) against the host reference of tests/approx_reference.py, which reads the text and the set of indexed
positions alone.

CPU tests tie the reference to a hand-worked table and to a brute force over every Hamming neighbour.  GPU tests
compare every match (its string, mismatches and occurrence set, and the byte order) over the spec matrix of
tests/test_kmers.py, k = 0..3; k = 0 against index_locate; hits and extract on the matches; the sliced path under a
node budget of 1, 7 and 4096; every golden file; argument errors; and a 16 M DNA text with planted near-copies."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES
import approx_reference as R
from index_matrix import IndexMatrix, device_index
from test_kmers import SPECS

EXPECTED = GOLDEN / "expected"

# ------------------------------------------------------------------ CPU: the reference itself
# three records ACGT% ACGA% TTGA$: Z = {'%', '$'}
T3, S3 = b"ACGT%ACGA%TTGA$", [0, 5, 10]
HAND = [
    # (text, starts, indexed (None: every position), query, k, cap, [(w, mismatches, positions)])
    (T3, S3, None, b"ACG", 0, 0, [(b"ACG", 0, [0, 5])]),
    (T3, S3, None, b"CGT", 1, 0, [(b"CGA", 1, [6]), (b"CGT", 0, [1])]),
    (T3, S3, None, b"CG%", 1, 0, [(b"CGA", 1, [6]), (b"CGT", 1, [1])]),   # a separator in the query
    (T3, S3, None, b"GA%", 1, 0, [(b"GA%", 0, [7]), (b"GT%", 1, [2])]),   # GA$: '$' is never substituted in
    (T3, S3, None, b"GA$", 1, 0, [(b"GA$", 0, [12])]),
    (T3, S3, None, b"AT", 1, 0, [(b"AC", 1, [0, 5]), (b"GT", 1, [2]), (b"TT", 1, [10])]),
    (T3, S3, None, b"AC", 2, 0, [(b"AC", 0, [0, 5]), (b"CG", 2, [1, 6]), (b"GA", 2, [7, 12]), (b"GT", 2, [2]),
                                 (b"TG", 2, [11]), (b"TT", 2, [10])]),
    (T3, S3, None, b"", 2, 0, []),
    (T3, S3, None, b"A" * 16, 16, 0, []),                                 # longer than the text
    (T3, S3, None, b"ACGA", 0, 2, [(b"AC", 0, [0, 5])]),                  # cap 2: m' = 2
    (T3, S3, set(range(15)) - {5}, b"ACG", 0, 0, [(b"ACG", 0, [0])]),     # position 5 not indexed
    (b"BANANA$", [0], None, b"NAN", 1, 0, [(b"BAN", 1, [0]), (b"NAN", 0, [2])]),   # ANA: 2 mismatches
]


@pytest.mark.parametrize("row", range(len(HAND)))
def test_reference_hand_worked(row):
    text, starts, indexed, q, k, cap, want = HAND[row]
    indexed = range(len(text)) if indexed is None else indexed
    assert R.matches(text, indexed, q, k, cap, starts) == want
    assert R.brute_force(text, indexed, q, k, cap, starts) == want


def test_reference_against_brute_force():
    """On 30 random tiny texts the sliding window and the neighbour enumeration give the same matches."""
    rng = random.Random(3)
    for trial in range(30):
        alpha = b"ACGT" if trial % 2 else b"AB%"
        n = rng.randrange(1, 30)
        text = bytes(rng.choice(alpha) for _ in range(n)) + b"$"
        starts = [0] + sorted(rng.sample(range(1, n + 1), min(n, rng.randrange(0, 3))))
        indexed = [p for p in range(len(text)) if trial % 3 or text[p] != ord("A")]
        cap = rng.choice([0, 0, 3])
        for _ in range(6):
            m = rng.randrange(0, 7)
            if m and rng.random() < 0.5 and m <= len(text):
                p = rng.randrange(0, len(text) - m + 1)
                q = text[p:p + m]
            else:
                q = bytes(rng.choice(alpha + b"$") for _ in range(m))
            for k in range(3):
                assert R.matches(text, indexed, q, k, cap, starts) == R.brute_force(text, indexed, q, k, cap, starts), \
                    (text, starts, q, k, cap)


# ------------------------------------------------------------------ GPU
def make_queries(text, starts, k, cap, seed):
    """Text substrings with 0..k+1 substitutions, random strings, queries with separators, lengths 1..40, longer than
    the cap, empty, and longer than the text."""
    rng = random.Random(seed)
    n = len(text)
    alphabet = sorted(set(text))
    z = sorted(R.separators(text, starts))
    qs = [b"", text + b"A"]
    for _ in range(60):
        m = rng.randrange(1, 41)
        if rng.random() < 0.75 and m <= n:
            p = rng.randrange(0, n - m + 1)
            q = bytearray(text[p:p + m])
            for j in rng.sample(range(m), min(m, rng.randrange(0, k + 2))):
                q[j] = rng.choice(alphabet)
            if rng.random() < 0.1 and z:
                q[rng.randrange(m)] = rng.choice(z)
            qs.append(bytes(q))
        else:
            qs.append(bytes(rng.choice(alphabet) for _ in range(m)))
    if cap:
        qs += [text[:cap + 3], text[1:cap + 9]]
    return qs


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


class Case(IndexMatrix):
    def __init__(self, S, name, tmp):
        (text, starts, names), flags, sources = SPECS[name]
        super().__init__(S, name, text, starts, names, flags, sources, tmp)
        self.text = text
        self.cap = flags.get("max_query_len") or 0


@pytest.fixture(scope="module", params=list(SPECS))
def case(request, S, tmp_path_factory):
    c = Case(S, request.param, tmp_path_factory.mktemp("approx"))
    yield c
    c.close()


def check_approx(index, text, starts, cap, queries, k):
    """Every match of every query against the reference: its string w (which also gives the byte order), its
    mismatches and its occurrences SA[rank_begin:rank_end] as a set."""
    sa = index.suffixes(0, index._s)
    got = index.approx_matches(queries, k)
    assert len(got) == len(queries)
    for q, rows in zip(queries, got):
        m = R.match_len(len(q), cap)
        have = [(text[int(sa[b]):int(sa[b]) + m], e, sorted(sa[b:en].tolist())) for e, b, en in rows]
        assert have == R.matches(text, sa, q, k, cap, starts), (q, k)
    return got


@pytest.mark.gpu
def test_approx_matches_reference(case, S):
    for label, index in case.indexes:
        for k in range(4):
            check_approx(index, case.text, case.starts, case.cap, make_queries(case.text, case.starts, k, case.cap, k), k)


@pytest.mark.gpu
def test_approx_k0_is_locate(case, S):
    for label, index in case.indexes:
        qs = [q for q in make_queries(case.text, case.starts, 0, case.cap, 7) if q]
        b, e, _ = index.locate_ranges(qs)
        got = index.approx_matches(qs, 0)
        for i, rows in enumerate(got):
            if b[i] == 0xFFFFFFFFFFFFFFFF:
                assert rows == [], qs[i]
            else:
                assert rows == [(0, int(b[i]), int(e[i]))], qs[i]


@pytest.mark.gpu
def test_approx_hits_extract_and_state(case, S):
    L = S._lib.lib()
    for label, index in case.indexes:
        k = 2
        qs = make_queries(case.text, case.starts, k, case.cap, 11)
        sa = index.suffixes(0, index._s)
        want = [R.matches(case.text, sa, q, k, case.cap, case.starts) for q in qs]
        got = index.locate_approx(qs, k)
        for q, rows, ref in zip(qs, got, want):
            assert [(e, sorted(h[0] for h in hits)) for e, hits in rows] == [(e, ps) for _, e, ps in ref], q
        # extract: prefix 0, suffix m' gives w for every hit of every match, in match order
        mis, rb, re_, ho, mo = index._approx(qs, k)
        total = int(ho[-1])
        if total:
            longest = max(R.match_len(len(q), case.cap) for q in qs if R.match_len(len(q), case.cap) <= len(case.text))
            (suf, _, _, _, offs), data = index.extract_window(0, total, 0, longest, 1 << 24)
            assert len(suf) == total
            strings = [data[int(offs[h]):int(offs[h + 1])] for h in range(total)]
            h = 0
            for qi, q in enumerate(qs):
                m = R.match_len(len(q), case.cap)
                for j in range(int(mo[qi]), int(mo[qi + 1])):
                    w = case.text[int(sa[rb[j]]):int(sa[rb[j]]) + m]
                    for _ in range(int(ho[j]), int(ho[j + 1])):  # (a region stops at its record's end)
                        got_w = strings[h]
                        assert got_w[:m] == w if len(got_w) >= m else w.startswith(got_w), (q, h)
                        h += 1
        # a window of the matches; then index_locate replaces the state
        cnt = len(mis)
        out = [np.zeros(max(1, cnt), np.uint64) for _ in range(3)] + [np.zeros(cnt + 1, np.uint64)]
        if cnt:
            assert L.sufr_b200_index_approx_matches(index._h, 1, cnt - 1, None, out[1].ctypes.data, None,
                                                    out[3].ctypes.data) == 0
            assert np.array_equal(out[1][:cnt - 1], rb[1:]) and np.array_equal(out[3][:cnt], ho[1:])
        assert L.sufr_b200_index_approx_matches(index._h, 0, cnt + 1, *[o.ctypes.data for o in out]) == \
            S._lib.ERR_ARGUMENT
        b, e, lho = index.locate_ranges(qs[2:4])
        assert index.hits(0, int(lho[-1]))[0].size == int(lho[-1])
        assert L.sufr_b200_index_approx_matches(index._h, 0, 0, None, None, None, out[3].ctypes.data) == \
            S._lib.ERR_ARGUMENT


@pytest.mark.gpu
@pytest.mark.parametrize("budget", ["1", "7", "4096"])
def test_approx_sliced(case, S, budget, monkeypatch):
    """A node budget smaller than a level: the sliced path gives the same matches, and the same per-level profile."""
    index = case.indexes[0][1]
    qs = make_queries(case.text, case.starts, 3, case.cap, 5)
    want = index.approx_matches(qs, 3)
    levels = index.approx_levels()
    monkeypatch.setenv("SUFR_B200_DEBUG_APPROX_NODES", budget)
    assert index.approx_matches(qs, 3) == want
    got_levels = index.approx_levels()
    assert all(np.array_equal(a, b) for a, b in zip(got_levels, levels))


@pytest.mark.gpu
@pytest.mark.parametrize("golden", [g for g, _, _ in GOLDEN_CASES])
def test_approx_golden(golden, S):
    index = S.SufrIndex.open(EXPECTED / golden)
    try:
        info = index.info
        text = index.string_at(0)
        qs = [text[p:p + 12] for p in range(0, len(text) - 12, max(1, len(text) // 20))]
        if info["seed_mask"] is not None:
            _, _, ho = index.locate_ranges(qs[:3])
            before = [x.tolist() for x in index.hits(0, int(ho[-1]))]
            with pytest.raises(S.SufrError) as e:
                index.approx_matches(qs, 1)
            assert e.value.code == S._lib.ERR_UNSUPPORTED
            assert [x.tolist() for x in index.hits(0, int(ho[-1]))] == before
            return
        cap = info["max_query_len"] or 0
        for k in (0, 1, 2):
            check_approx(index, text, info["sequence_starts"], cap, qs, k)
    finally:
        index.close()


@pytest.mark.gpu
def test_approx_argument_errors(S):
    index, r = device_index(S, b"ACGTACGTTTGA$", None, None)
    try:
        L = S._lib.lib()
        blob = np.frombuffer(b"ACGTAC", np.uint8)
        offs = np.array([0, 3, 6], np.uint64)
        bad_offs = np.array([0, 4, 3], np.uint64)
        mo = np.zeros(3, np.uint64)
        hits = C.c_uint64()
        h, E = index._h, S._lib.ERR_ARGUMENT
        assert L.sufr_b200_index_approx_matches(h, 0, 0, None, None, None, None) == E  # before any approx
        calls = [
            lambda: L.sufr_b200_index_approx(None, blob.ctypes.data, offs.ctypes.data, 2, 1, mo.ctypes.data, C.byref(hits)),
            lambda: L.sufr_b200_index_approx(h, None, offs.ctypes.data, 2, 1, mo.ctypes.data, C.byref(hits)),
            lambda: L.sufr_b200_index_approx(h, blob.ctypes.data, None, 2, 1, mo.ctypes.data, C.byref(hits)),
            lambda: L.sufr_b200_index_approx(h, blob.ctypes.data, offs.ctypes.data, 2, 1, None, C.byref(hits)),
            lambda: L.sufr_b200_index_approx(h, blob.ctypes.data, offs.ctypes.data, 2, 1, mo.ctypes.data, None),
            lambda: L.sufr_b200_index_approx(h, blob.ctypes.data, bad_offs.ctypes.data, 2, 1, mo.ctypes.data,
                                             C.byref(hits)),
            lambda: L.sufr_b200_index_approx(h, blob.ctypes.data, offs.ctypes.data, 2, 17, mo.ctypes.data, C.byref(hits)),
        ]
        for f in calls:
            assert f() == E
        assert L.sufr_b200_index_approx(h, blob.ctypes.data, offs.ctypes.data, 2, 16, mo.ctypes.data,
                                        C.byref(hits)) == 0
        assert int(mo[-1]) > 0 and hits.value > 0
        assert L.sufr_b200_index_approx_matches(h, int(mo[-1]), 1, None, None, None, None) == E
        assert L.sufr_b200_index_approx_matches(h, int(mo[-1]), 0, None, None, None, None) == 0
        with pytest.raises(S.SufrError):
            index.approx_matches([b"ACG"], -1)
        assert index.approx_matches([], 2) == []
    finally:
        index.close()
        r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [32, 64])
def test_approx_16M_planted(bits, S):
    """A 16 M DNA text with near-copies of the queries planted in it, checked by a numpy sliding window at k <= 3."""
    import torch
    rng = np.random.default_rng(21)
    n = 1 << 24
    t = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    qs = []
    for i in range(6):
        q = t[rng.integers(0, n - 20, 1)[0]:][:20].copy()
        qs.append(q.tobytes())
        for e in range(5):  # copies with e substitutions
            c = q.copy()
            for j in rng.choice(20, e, replace=False):
                c[j] = np.frombuffer(b"ACGT", np.uint8)[(b"ACGT".index(bytes([c[j]])) + 1) % 4]
            at = int(rng.integers(0, n - 20))
            t[at:at + 20] = c
    t[rng.integers(0, n, 3000)] = ord("N")
    t[-1] = ord("$")
    starts = [0, n // 2]
    t[n // 2 - 1] = ord("%")
    text = t.tobytes()
    dt = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", is_dna=True, sequence_starts=starts, sequence_names=["a", "b"])
    r = S.build(args, index_bits=bits, result_memory=S.MEM_DEVICE, device_text=(dt.data_ptr(), dt.numel()))
    index = S.SufrIndex(r, args)
    try:
        indexed = np.zeros(n, bool)
        indexed[index.suffixes(0, index._s).astype(np.int64)] = True
        got = {k: index.locate_approx(qs, k) for k in range(4)}
        for i, q in enumerate(qs):
            qa = np.frombuffer(q, np.uint8)
            mis = np.zeros(n - 19, np.int64)
            bad = np.zeros(n - 19, bool)
            for j in range(20):
                c = t[j:n - 19 + j]
                d = c != qa[j]
                mis += d
                bad |= d & ((c == ord("$")) | (c == ord("%")))
            for k in range(4):
                pos = np.flatnonzero((mis <= k) & ~bad & indexed[:n - 19])
                rows = got[k][i]
                assert sorted(p for _, hits in rows for p, _, _ in hits) == pos.tolist(), (k, q)
                assert all(e == int(mis[p]) for e, hits in rows for p, _, _ in hits)
                assert len(rows) == len({text[p:p + 20] for p in pos.tolist()})
    finally:
        index.close()
        r.free()
