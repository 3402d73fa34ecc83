"""Matching statistics and maximal exact matches on a device index (`matching_stats_kernel`, sufr_b200_index_matching_stats
/ _mems, SufrIndex.matching_statistics / .mems / .locate_mems) against the host reference of tests/mems_reference.py.

CPU tests tie the reference to a hand-worked table and to a literal all-pairs enumeration of MEMs.  GPU tests compare
every position of every query over a matrix of index sources (device builds, written and reopened files; u32 and u64),
modes (plain, DNA, DNA with ambiguity, build caps 2, 5, 12 and 32) and sizes (1 suffix to 64 KB), check a 2 M text
through the existing search, and check the hits and regions that index_hits / index_extract return after index_mems."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES
import mems_reference as M
import search_reference as R
from sufrfile import parse_sufr
from test_extract import concat_windows, restate_region
from test_search_reference import ACGT, PROTEIN, WIDE, make_text

EXPECTED = GOLDEN / "expected"
NONE = M.NONE


# ------------------------------------------------------------------ CPU: the reference itself
# (text, SA, build cap) and rows (query, ms, rank_begin, rank_end, MEMs with min_len 1)
HAND = {
    "banana": ((b"BANANA", [5, 3, 1, 0, 4, 2], 0), [
        # ANA occurs at 3 and 1 (ranks 1, 2); NA at 4, 2; A everywhere it starts a suffix; B once
        (b"ANAB", [3, 2, 1, 1], [(1, 3), (4, 6), (0, 3), (3, 4)], [(0, 3, 1, 3), (3, 1, 3, 4)]),
        (b"XNAN", [0, 3, 2, 1], [None, (5, 6), (1, 3), (4, 6)], [(1, 3, 5, 6)]),
        (b"BANANAS", [6, 5, 4, 3, 2, 1, 0], [(3, 4), (2, 3), (5, 6), (1, 3), (4, 6), (0, 3), None],
         [(0, 6, 3, 4)]),
        (b"", [], [], []),
    ]),
    # ABABAB uncapped: SA AB(4) ABAB(2) ABABAB(0) B(5) BAB(3) BABAB(1); ms falls by one per position, one MEM
    "ababab": ((b"ABABAB", [4, 2, 0, 5, 3, 1], 0), [
        (b"ABABX", [4, 3, 2, 1, 0], [(1, 3), (4, 6), (0, 3), (3, 6), None], [(0, 4, 1, 3)]),
    ]),
    # the same text built with cap 2 (the same array): every length stops at 2, so three MEMs of "at least 2"
    "ababab_q2": ((b"ABABAB", [4, 2, 0, 5, 3, 1], 2), [
        (b"ABABX", [2, 2, 2, 1, 0], [(0, 3), (4, 6), (0, 3), (3, 6), None], [(0, 2, 0, 3), (1, 2, 4, 6), (2, 2, 0, 3)]),
        (b"BB", [1, 1], [(3, 6), (3, 6)], [(0, 1, 3, 6), (1, 1, 3, 6)]),
    ]),
}


@pytest.mark.parametrize("name", list(HAND))
def test_reference_hand_worked(name):
    import oracle as O
    (text, sa, cap), rows = HAND[name]
    _, spec_sa, spec_lcp = O.spec_build(text, max_query_len=cap or None)
    assert spec_sa == sa  # the table's array is that of the index definition
    m = M.Matcher(R.Index(text, np.array(sa), np.array(spec_lcp), cap))
    for q, ms, ranges, mems in rows:
        got_ms, b, e = m.stats(q)
        assert got_ms.tolist() == ms, q
        assert [None if x == NONE else (int(x), int(y)) for x, y in zip(b, e)] == ranges, q
        assert M.mems_of(got_ms, b, e, 1) == mems, q


def test_reference_against_all_pairs_mems():
    """On small random uncapped plain indexes: ms[i] is the longest match over all pairs, every listed occurrence is a
    literal MEM (maximal both ways), and at a MEM start the listed occurrences are exactly the literal MEMs of length
    ms[i] there."""
    rng = random.Random(3)
    for trial in range(30):
        alpha = b"AC" if trial % 3 == 0 else (b"ACGT" if trial % 3 == 1 else b"AB$")
        n = rng.randrange(1, 60)
        text = bytes(rng.choice(alpha) for _ in range(n))
        sa = sorted(range(n), key=lambda p: text[p:])
        idx = R.Index(text, np.array(sa), np.zeros(n, np.int64))
        m = M.Matcher(idx)
        for _ in range(6):
            if rng.random() < 0.5 and n > 1:
                p = rng.randrange(n)
                q = bytearray(text[p:p + rng.randrange(1, 40)])
                for k in range(len(q)):
                    if rng.random() < 0.15:
                        q[k] = rng.choice(alpha + b"X")
                q = bytes(q)
            else:
                q = bytes(rng.choice(alpha + b"X") for _ in range(rng.randrange(0, 30)))
            ms, b, e = m.stats(q)
            for i in range(len(q)):
                best = max((next((k for k in range(min(len(q) - i, n - p)) if q[i + k] != text[p + k]),
                                 min(len(q) - i, n - p)) for p in range(n)), default=0)
                assert ms[i] == best, (text, q, i)
            for L in (1, 2, 3, 5):
                mems = M.mems_of(ms, b, e, L)
                listed = M.occurrences(idx, mems)
                literal = M.literal_mems(text, set(range(n)), q, L)
                assert listed <= literal, (text, q, L, sorted(listed - literal)[:5])
                for i, ln, _, _ in mems:
                    assert {x for x in listed if x[0] == i} == {x for x in literal if x[0] == i and x[2] == ln}
                assert all(ln <= ms[i] for i, _, ln in literal)


# ------------------------------------------------------------------ GPU fixtures
def with_records(text, k, seed):
    """`text` with k - 1 of its bytes replaced by the delimiter '%': (text, sequence starts, names)."""
    n = len(text)
    if k <= 1 or n < 4 * k:
        return text, [0], ["r0"]
    rng = random.Random(seed)
    cut = sorted(rng.sample(range(1, n - 2), k - 1))
    t = bytearray(text)
    for c in cut:
        t[c] = ord("%")
    return bytes(t), [0] + [c + 1 for c in cut], [f"r{i}" for i in range(k)]


ALL = [("built", 32), ("built", 64), ("file", 32), ("file", 64)]
SPECS = {
    # name -> (text, starts, names), build flags, index sources
    "tiny_1": ((b"NNNA", [0], ["r0"]), dict(is_dna=True), ALL),
    "tiny_q2": ((b"NAAA", [0], ["r0"]), dict(is_dna=True, max_query_len=2), ALL),
    "acgt_plain_4k": (with_records(make_text(41, 4000, ACGT, copies=40, runs=[(b"T", 40)]), 8, 1), dict(), ALL),
    "dna_N_4k": (with_records(make_text(42, 4000, ACGT, copies=40, runs=[(b"T", 30)], rare=b"N", rare_p=0.01), 8, 2),
                 dict(is_dna=True), ALL),
    "dna_N_amb_4k": (with_records(make_text(42, 4000, ACGT, copies=40, runs=[(b"T", 30)], rare=b"N", rare_p=0.01), 8,
                                  2), dict(is_dna=True, allow_ambiguity=True), ALL),
    "dna_q2_4k": (with_records(make_text(43, 4000, ACGT, copies=40), 4, 3), dict(is_dna=True, max_query_len=2), ALL),
    "protein_q5": (with_records(make_text(44, 5000, PROTEIN, copies=80), 6, 4), dict(max_query_len=5), ALL),
    "protein_q12_nodollar": (with_records(make_text(45, 5000, PROTEIN, copies=80, dollar=False), 6, 5),
                             dict(max_query_len=12), ALL),
    "dna_q32": (with_records(make_text(46, 6000, ACGT, copies=60, copy_len=(30, 200), runs=[(b"AC", 50)]), 6, 6),
                dict(is_dna=True, max_query_len=32), ALL),
    "wide_nodollar": (with_records(make_text(47, 3000, WIDE, copies=30, dollar=False), 4, 7), dict(), ALL),
    "dna_64k": (with_records(make_text(48, 64_000, ACGT, copies=100, copy_len=(20, 2000), runs=[(b"T", 200)],
                                       rare=b"N", rare_p=0.0005), 16, 8), dict(is_dna=True),
                [("built", 32), ("file", 64)]),
    "protein_64k_q12": (with_records(make_text(49, 64_000, PROTEIN, copies=200, copy_len=(12, 300)), 16, 9),
                        dict(max_query_len=12), [("built", 64), ("file", 32)]),
}


def make_queries(text, starts, seed, alphabet, whole=True):
    """Reads with substitutions, reads across record delimiters, bytes the text lacks, queries longer than the text,
    the whole text and empty queries, in one mixed batch."""
    rng = random.Random(seed)
    n = len(text)
    qs = []
    for _ in range(60):  # substrings of the text with random substitutions
        p = rng.randrange(n)
        q = bytearray(text[p:p + rng.randrange(1, 160)])
        rate = rng.choice([0.0, 0.01, 0.03, 0.1])
        for k in range(len(q)):
            if rng.random() < rate:
                q[k] = rng.choice(alphabet)
        qs.append(bytes(q))
    for s in starts[1:][:10]:  # across a record delimiter
        qs.append(text[max(0, s - rng.randrange(2, 60)):s + rng.randrange(1, 60)])
    qs += [b"\x01", b"\xff\xfe", b"acgt", b"A\xffC" + text[:20], b"%", b"$", b"\x00A"]  # bytes the text lacks
    qs += [bytes(rng.choice(alphabet) for _ in range(rng.randrange(1, 80))) for _ in range(10)]
    qs += [b"", b""]
    tail = text[max(0, n - 30):]
    qs += [tail + b"A", tail + tail, text[:40] + b"\x01" + text[:40]]  # past the end of the text
    if whole:
        qs += [text, text + b"A" + text[:50]]  # the whole text; longer than the text
    qs.insert(len(qs) // 2, b"")
    return qs


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


class Case:
    """One text built every way its spec lists, its reference matcher and queries."""

    def __init__(self, S, name, tmp):
        import torch
        (text, starts, names), flags, sources = SPECS[name]
        self.name, self.flags, self.starts, self.names = name, flags, starts, names
        self.indexes, self._results, arrays = [], [], None
        try:
            for kind, bits in sources:
                if kind == "built":
                    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
                    args = S.SufrBuilderArgs(text=b"", sequence_starts=starts, sequence_names=names, **flags)
                    r = S.build(args, index_bits=bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
                    r._keep = t
                    self._results.append(r)
                    udt = np.uint32 if bits == 32 else np.uint64
                    got = (r.text_tensor().cpu().numpy().tobytes(), r.sa_tensor().cpu().numpy().view(udt),
                           r.lcp_tensor().cpu().numpy().view(udt))
                    index = S.SufrIndex(r, args)
                else:
                    path = tmp / f"{name}_u{bits}.sufr"
                    b = S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(path), sequence_starts=starts,
                                                        sequence_names=names, **flags), bits)
                    b._res.free()
                    f = parse_sufr(path.read_bytes())
                    assert f.index_bits == bits
                    got = (f.text, f.sa, f.lcp)
                    index = S.SufrIndex.open(path)
                self.indexes.append((f"{kind}_u{bits}", index))
                got = (got[0], got[1].astype(np.int64), got[2].astype(np.int64))
                if arrays is None:
                    arrays = got
                else:
                    assert got[0] == arrays[0] and np.array_equal(got[1], arrays[1]) and np.array_equal(got[2], arrays[2])
        except BaseException:
            self.close()
            raise
        self.ref = R.Index(arrays[0], arrays[1], arrays[2], flags.get("max_query_len") or 0)
        self.text = arrays[0]
        self.matcher = M.Matcher(self.ref)
        alphabet = sorted(set(text)) or [65]
        self.queries = make_queries(self.text, starts, name, alphabet, whole=len(text) <= 8000)
        self.want = M.expected_stats(self.matcher, self.queries)
        self.cap = flags.get("max_query_len") or 0

    def min_lens(self):
        top = max([int(w[0].max()) for w in self.want if len(w[0])] or [0])
        lens = [1, 2, top + 1]
        if self.cap:
            lens += [self.cap - 1, self.cap, self.cap + 1]
        else:
            lens += [12, 20]
        return sorted({x for x in lens if x >= 1})

    def want_mems(self, min_len):
        return [M.mems_of(*w, min_len) for w in self.want]

    def close(self):
        for _, index in self.indexes:
            index.close()
        for r in self._results:
            r.free()
        self.indexes, self._results = [], []


@pytest.fixture(scope="module", params=list(SPECS))
def case(request, S, tmp_path_factory):
    c = Case(S, request.param, tmp_path_factory.mktemp("mems"))
    yield c
    c.close()


def as_lists(stats):
    return [tuple(np.asarray(c, np.uint64) for c in s) for s in stats]


# ------------------------------------------------------------------ GPU: the matrix against the reference
@pytest.mark.gpu
def test_matching_statistics_match_reference(case):
    for label, index in case.indexes:
        got = index.matching_statistics(case.queries)
        bad = M.first_mismatch(got, case.want, case.queries)
        assert bad is None, f"{case.name} {label}: {bad}"


@pytest.mark.gpu
def test_mems_match_reference(case):
    for label, index in case.indexes:
        for L in case.min_lens():
            want = case.want_mems(L)
            got = index.mems(case.queries, L)
            assert got == [[w[:4] for w in ws] for ws in want], f"{case.name} {label} min_len={L}"
            if L == max(case.min_lens()):
                assert got == [[] for _ in case.queries]  # larger than every match


def restate_hits(ref, starts, mems):
    """(suffix, sequence, sequence_pos) of every occurrence of the MEMs, in MEM order then rank order."""
    st = np.asarray(starts, dtype=np.int64)
    suf = np.asarray([int(ref.sa[r]) for _, _, b, e in mems for r in range(b, e)], dtype=np.int64)
    seq = np.searchsorted(st, suf, side="right") - 1
    return suf, seq, suf - st[seq]


@pytest.mark.gpu
def test_hits_and_extract_after_mems(case):
    """index_hits / index_extract after index_mems return the MEMs' occurrences: equal to a numpy restatement, in
    windows and with the zero-entry retry of a region larger than the byte budget."""
    L = case.cap if 0 < case.cap < 8 else 8
    # a leading run of the batch with at most 20 000 occurrences, so the windows stay few
    qs, wants, hits = [], [], 0
    for q, w in zip(case.queries, case.want):
        mems = M.mems_of(*w, L)
        hits += sum(e - b for _, _, b, e in mems)
        if hits > 20_000 and qs:
            break
        qs.append(q)
        wants.append(mems)
    flat = [m for ws in wants for m in ws]
    counts = [e - b for _, _, b, e in flat]
    want_suf, want_seq, want_pos = restate_hits(case.ref, case.starts, flat)
    for label, index in case.indexes:
        q, p, ln, b, e, ho = index._mems(qs, L)
        assert list(zip(p.tolist(), ln.tolist(), b.tolist(), e.tolist())) == [m for m in flat], label
        assert q.tolist() == [k for k, ws in enumerate(wants) for _ in ws], label
        assert ho.tolist() == [0] + np.cumsum(counts, dtype=np.int64).tolist(), label
        total = int(ho[-1])
        suf, seq, pos = index.hits(0, total)
        assert suf.tolist() == want_suf.tolist() and seq.tolist() == want_seq.tolist(), label
        assert pos.tolist() == want_pos.tolist(), label
        if total:
            mid = total // 2
            assert index.hits(mid, total - mid)[0].tolist() == want_suf[mid:].tolist()
        for P, S_, budget, upto in ((3, 5, 7, 300), (None, None, 50, 300), (0, 1, 1 << 20, total)):
            part = min(upto, total)
            if part == 0:
                assert index.extract_window(0, 0, P, S_)[1] == b""
                continue
            cols, sizes, data = concat_windows(index, part, 13 if part < total else 4096, P, S_, budget)
            regions = [restate_region(case.text, case.starts, int(s), P, S_) for s in want_suf[:part]]
            assert cols[0].tolist() == want_suf[:part].tolist(), (label, P, S_)
            assert [(x[1], x[2]) for x in regions] == list(zip(cols[2].tolist(), cols[3].tolist())), (label, P, S_)
            assert data == b"".join(x[4] for x in regions), (label, P, S_)
        located = index.locate_mems(qs, L)
        assert [[(qp, ml) for qp, ml, _ in ws] for ws in located] == [[m[:2] for m in ws] for ws in wants], label
        got_hits = [h for ws in located for _, _, hs in ws for h in hs]
        names = case.names
        assert got_hits == [(int(s), names[int(k)], int(x)) for s, k, x in zip(want_suf, want_seq, want_pos)], label


# ------------------------------------------------------------------ GPU: goldens, 2 M text, state, errors
@pytest.mark.gpu
@pytest.mark.parametrize("golden", [c[0] for c in GOLDEN_CASES])
def test_goldens(S, golden):
    """Every golden file: the reference's answers, or ERR_UNSUPPORTED for a seed-mask index; locate stays right."""
    f = parse_sufr((EXPECTED / golden).read_bytes())
    ref = R.Index(f.text, f.sa, f.lcp, 0 if f.seed_mask else f.max_query_len, f.seed_mask)
    rng = random.Random(golden)
    text = f.text
    queries = [text[p:p + rng.randrange(1, 80)] for p in (rng.randrange(len(text)) for _ in range(30))]
    queries += [text[:3000], b"ZZ" + text[:30], b"", text[-5:] + b"AC"]
    idx = S.SufrIndex.open(EXPECTED / golden)
    try:
        if f.seed_mask:
            for call in (lambda: idx.matching_statistics(queries), lambda: idx.mems(queries, 3)):
                with pytest.raises(S.SufrError) as ei:
                    call()
                assert ei.value.code == 5 and "seed mask" in str(ei.value)
        else:
            want = M.expected_stats(M.Matcher(ref), queries)
            assert M.first_mismatch(idx.matching_statistics(queries), want, queries) is None
            assert idx.mems(queries, 3) == [M.mems_of(*w, 3) for w in want]
        short = [q[:6] for q in queries]
        b, e, _ = idx.locate_ranges(short, low_memory=True)
        got = [None if x == NONE else (int(x), int(y)) for x, y in zip(b, e)]
        assert got == R.full_ranges(ref, short)
    finally:
        idx.close()


@pytest.mark.gpu
def test_2m_text_through_search(S, tmp_path):
    """A 2 M text: every position checked through the existing search.  count(q[i, i+ms)) = re - rb (the whole
    range equals search's), q[i, i+ms+1) occurs nowhere, and the range's first and last suffixes start with q[i, i+ms)."""
    import torch
    text = make_text(9, 2_000_000, ACGT, copies=300, copy_len=(1000, 20000), runs=[(b"T", 3000)])
    flags = dict(is_dna=True)
    path = tmp_path / "2m_u64.sufr"
    S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(path), **flags), 64)._res.free()
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", **flags)
    r = S.build(args, index_bits=32, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    built, opened = S.SufrIndex(r, args), S.SufrIndex.open(path)
    try:
        sa = r.sa_tensor().cpu().numpy().view(np.uint32).astype(np.int64)
        rng = random.Random(2)
        qs = []
        for _ in range(100):
            p = rng.randrange(len(text) - 200)
            q = bytearray(text[p:p + 150])
            for k in range(len(q)):
                if rng.random() < 0.01:
                    q[k] = rng.choice(b"ACGT")
            qs.append(bytes(q))
        qs += [bytes(rng.choice(b"ACGTN") for _ in range(150)) for _ in range(20)]
        qs += [text[500_000:502_000], b"", b"T" * 4000]
        stats = built.matching_statistics(qs)
        assert M.first_mismatch(opened.matching_statistics(qs), stats, qs) is None
        subs, ranges, longer = [], [], []
        for q, (ms, b, e) in zip(qs, stats):
            for i in range(len(q)):
                k = int(ms[i])
                if k:
                    subs.append(q[i:i + k])
                    ranges.append((int(b[i]), int(e[i])))
                    lo, hi = sa[int(b[i])], sa[int(e[i]) - 1]
                    assert text[lo:lo + k] == q[i:i + k] and text[hi:hi + k] == q[i:i + k]
                else:
                    assert b[i] == NONE and e[i] == NONE
                if i + k < len(q):
                    longer.append(q[i:i + k + 1])
        assert built.search(subs, low_memory=True) == ranges
        assert all(x is None for x in built.search(longer, low_memory=True))
        assert len(subs) > 10_000
    finally:
        built.close()
        opened.close()
        r.free()


@pytest.mark.gpu
def test_locate_mems_extract_state(S):
    """locate -> mems -> extract -> locate -> extract: hits and extract read the state of the latest call."""
    (text, starts, names), flags, _ = SPECS["acgt_plain_4k"]
    f_ref = R.Index(text, np.array(sorted(range(len(text)), key=lambda p: text[p:])), np.zeros(len(text), np.int64))
    import torch
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", sequence_starts=starts, sequence_names=names, **flags)
    r = S.build(args, index_bits=32, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    idx = S.SufrIndex(r, args)
    try:
        sa = r.sa_tensor().cpu().numpy().view(np.uint32).astype(np.int64)
        assert sa.tolist() == f_ref.sa.tolist()
        locq = [text[100:110], text[7:10]]
        memq = [text[200:260] + b"X" + text[900:930]]
        want_loc = sorted(sa[r0] for rr in R.full_ranges(f_ref, locq) for r0 in range(*rr))

        for step in range(2):
            b, e, ho = idx.locate_ranges(locq)
            assert sorted(idx.hits(0, int(ho[-1]))[0].tolist()) == want_loc
            mems = idx.mems(memq, 10)
            assert [(m[0], m[1]) for m in mems[0]] == [(0, 60), (61, 30)]
            want = sorted(int(sa[rk]) for m in mems[0] for rk in range(m[2], m[3]))
            arrs, data = idx.extract_window(0, len(want), 0, 4)
            assert sorted(arrs[0].tolist()) == want
            assert all(data[int(arrs[4][k]):int(arrs[4][k + 1])] == restate_region(text, starts, s, 0, 4)[4]
                       for k, s in enumerate(arrs[0].tolist()))
            b, e, ho = idx.locate_ranges(locq)
            arrs, _ = idx.extract_window(0, int(ho[-1]), 0, 3)
            assert sorted(arrs[0].tolist()) == want_loc
    finally:
        idx.close()
        r.free()


@pytest.mark.gpu
def test_argument_errors_and_empty_batches(S, tmp_path):
    from sufr_b200 import _lib
    L = _lib.lib()
    (text, starts, names), flags, _ = SPECS["dna_N_4k"]
    path = tmp_path / "e.sufr"
    S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(path), sequence_starts=starts, sequence_names=names,
                                    **flags), 32)._res.free()
    idx = S.SufrIndex.open(path)
    f = parse_sufr(path.read_bytes())
    matcher = M.Matcher(R.Index(f.text, f.sa, f.lcp))
    qs = [text[10:60], b"ACGTX" + text[300:340]]
    want = M.expected_stats(matcher, qs)
    try:
        blob, offs = idx._pack_queries(qs)
        total = int(offs[-1])
        out = [np.zeros(total + 1, np.uint64) for _ in range(6)]
        num = C.c_uint64()
        p = [o.ctypes.data for o in out]
        cases = [
            L.sufr_b200_index_matching_stats(None, blob.ctypes.data, offs.ctypes.data, 2, p[0], p[1], p[2]),
            L.sufr_b200_index_matching_stats(idx._h, None, offs.ctypes.data, 2, p[0], p[1], p[2]),
            L.sufr_b200_index_matching_stats(idx._h, blob.ctypes.data, None, 2, p[0], p[1], p[2]),
            L.sufr_b200_index_matching_stats(idx._h, blob.ctypes.data, offs.ctypes.data, 2, None, p[1], p[2]),
            L.sufr_b200_index_matching_stats(idx._h, blob.ctypes.data, offs.ctypes.data, 2, p[0], p[1], None),
            L.sufr_b200_index_mems(idx._h, blob.ctypes.data, offs.ctypes.data, 2, 0, C.byref(num), *p),
            L.sufr_b200_index_mems(idx._h, blob.ctypes.data, offs.ctypes.data, 2, 5, None, *p),
            L.sufr_b200_index_mems(idx._h, blob.ctypes.data, offs.ctypes.data, 2, 5, C.byref(num), None, *p[1:]),
            L.sufr_b200_index_mems(idx._h, blob.ctypes.data, offs.ctypes.data, 2, 5, C.byref(num), *p[:5], None),
            L.sufr_b200_index_mems(idx._h, None, offs.ctypes.data, 2, 5, C.byref(num), *p),
        ]
        assert cases == [_lib.ERR_ARGUMENT] * len(cases)
        bad = np.array([0, 30, 10], np.uint64)
        assert L.sufr_b200_index_matching_stats(idx._h, blob.ctypes.data, bad.ctypes.data, 2, *p[:3]) == _lib.ERR_ARGUMENT
        assert "ascending" in L.sufr_b200_last_error().decode()
        for bad_len in (0, -3):
            with pytest.raises(S.SufrError) as ei:
                idx.mems(qs, bad_len)
            assert ei.value.code == _lib.ERR_ARGUMENT
        assert M.first_mismatch(idx.matching_statistics(qs), want, qs) is None  # still answers
        assert idx.mems(qs, 5) == [M.mems_of(*w, 5) for w in want]
        # empty batches: no entries, no hits
        assert idx.matching_statistics([]) == []
        got = idx.matching_statistics([b"", b""])
        assert [len(x[0]) for x in got] == [0, 0]
        assert idx.mems([b"", b""], 3) == [[], []]
        assert idx.mems([], 3) == []
        assert idx.hits(0, 0)[0].tolist() == []
        assert idx.extract_window(0, 0)[1] == b""
        with pytest.raises(S.SufrError):
            idx.hits(0, 1)
        lm = idx.locate_mems(qs, 5)
        assert [[(a, b, len(h)) for a, b, h in ws] for ws in lm] == \
            [[(m[0], m[1], m[3] - m[2]) for m in M.mems_of(*w, 5)] for w in want]
    finally:
        idx.close()
    # a seed-mask index is refused, and still answers locate afterwards
    mpath = tmp_path / "mask.sufr"
    S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(mpath), seed_mask="1101", **flags), 32)._res.free()
    midx = S.SufrIndex.open(mpath)
    try:
        before = midx.locate_ranges(qs[:1])
        for call in (lambda: midx.matching_statistics(qs), lambda: midx.mems(qs, 4), lambda: midx.locate_mems(qs, 4)):
            with pytest.raises(S.SufrError) as ei:
                call()
            assert ei.value.code == _lib.ERR_UNSUPPORTED
        after = midx.locate_ranges(qs[:1])
        assert all(np.array_equal(x, y) for x, y in zip(before, after))
    finally:
        midx.close()
