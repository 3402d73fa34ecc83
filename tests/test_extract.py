"""extract, list and string_at on a device index (sufr_b200_index_extract / _list / _string_at, SufrIndex.extract /
.list / .string_at), checked field by field and byte by byte against a numpy restatement over the `.sufr` file
(tests/sufrfile.py) and the hits of SufrIndex.locate, which test_file_query.py pins to the reference's fixtures."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES, ROOT
from index_matrix import device_index
from sufrfile import parse_sufr

EXPECTED = GOLDEN / "expected"
U64_MAX = 0xFFFFFFFFFFFFFFFF


@pytest.fixture(scope="module")
def S():
    import subprocess
    subprocess.check_call(["make", "-C", str(ROOT / "sufr_b200" / "csrc"), "-s", "-j8"])
    import sufr_b200
    return sufr_b200


# ------------------------------------------------------------------ the restatement (pure numpy / Python)
def record_of(starts, n, p):
    """(record index or None, a, e): record i owns [s_i, s_{i+1}) and the last one [s_{k-1}, n); a position before
    the first start (or any position without starts) belongs to [0, s_0) (or [0, n)) and to no record."""
    i = int(np.searchsorted(np.asarray(starts, dtype=np.uint64), np.uint64(p), side="right")) - 1
    if i < 0:
        return None, 0, (starts[0] if len(starts) else n)
    return i, starts[i], (starts[i + 1] if i + 1 < len(starts) else n)


def restate_region(text, starts, p, prefix_len=None, suffix_len=None):
    """(record, start, end, suffix_offset, bytes) of the hit at suffix p (include/sufr_b200.h)."""
    i, a, e = record_of(starts, len(text), p)
    rel = p - a
    start = rel - min(rel, prefix_len or 0)
    end = e - a if suffix_len is None else min(rel + suffix_len, e - a)
    return i, start, end, rel - start, bytes(text[a + start:a + end])


def restate_extract(text, starts, names, located, prefix_len=None, suffix_len=None):
    """SufrIndex.extract restated from SufrIndex.locate's hits: per query a list of
    (rank, suffix, name, sequence_start, (start, end), suffix_offset, bytes)."""
    out = []
    for hits in located:
        rows = []
        for rank, suf, _, _ in hits:
            i, start, end, off, data = restate_region(text, starts, suf, prefix_len, suffix_len)
            rows.append((rank, suf, None if i is None else names[i], 0 if i is None else starts[i], (start, end), off,
                         data))
        out.append(rows)
    return out


def as_rows(results):
    return [[(e.rank, e.suffix, e.sequence_name, e.sequence_start, e.sequence_range, e.suffix_offset, e.sequence)
             for e in r.sequences] for r in results]


# ------------------------------------------------------------------ CPU
def test_restatement_on_the_hand_worked_table():
    f = parse_sufr((EXPECTED / "2.sufr").read_bytes())
    assert f.text == b"ACGTACGT%ACGTACGT$"
    assert f.sequence_starts == [0, 9] and f.sequence_names == ["ABC", "DEF"]
    hits = [15, 6, 11, 2]  # GT in rank order
    got = [restate_region(f.text, f.sequence_starts, p, 1, 2) for p in hits]
    assert got == [(1, 5, 8, 1, b"CGT"), (0, 5, 8, 1, b"CGT"), (1, 1, 4, 1, b"CGT"), (0, 1, 4, 1, b"CGT")]
    got = [restate_region(f.text, f.sequence_starts, p, 1, None) for p in hits[:2]]
    assert got == [(1, 5, 9, 1, b"CGT$"), (0, 5, 9, 1, b"CGT%")]
    located = [[(r, p, None, None) for r, p in zip(range(6, 10), hits)]]
    (rows,) = restate_extract(f.text, f.sequence_starts, f.sequence_names, located, 1, 2)
    assert [(x[0], x[2], x[3], x[4], x[5], x[6]) for x in rows] == [
        (6, "DEF", 9, (5, 8), 1, b"CGT"), (7, "ABC", 0, (5, 8), 1, b"CGT"), (8, "DEF", 9, (1, 4), 1, b"CGT"),
        (9, "ABC", 0, (1, 4), 1, b"CGT")]


def test_restatement_clipping():
    text, starts = b"ACGTACGT%ACGTACGT$", [0, 9]
    assert restate_region(text, starts, 8, 2, 5) == (0, 6, 9, 2, b"GT%")      # the delimiter belongs to its record
    assert restate_region(text, starts, 17, 0, None) == (1, 8, 9, 0, b"$")     # the final '$' too
    assert restate_region(text, starts, 6, 3, 0) == (0, 3, 6, 3, b"TAC")      # S = 0: only the prefix
    assert restate_region(text, starts, 6, 0, 0) == (0, 6, 6, 0, b"")
    assert restate_region(text, starts, 11, 5, 1) == (1, 0, 3, 2, b"ACG")     # P beyond the record start
    assert restate_region(text, starts, 11, 1000, None) == (1, 0, 9, 2, b"ACGTACGT$")
    assert restate_region(text, [3, 9], 1, 5, 1) == (None, 0, 2, 1, b"AC")    # before the first start: [0, s_0)
    assert restate_region(text, [], 12, 2, 100) == (None, 10, 18, 2, b"CGTACGT$")  # no starts: [0, n)


# ------------------------------------------------------------------ GPU helpers
PS = [(None, None), (0, 0), (0, 1), (3, 5), (1000, None)]


def golden_queries(f, seed):
    rng = random.Random(seed)
    text = f.text.decode("latin-1")
    qs = []
    for _ in range(40):
        p, ln = rng.randrange(len(text)), rng.randrange(1, 9)
        qs.append(text[p:p + ln])
    for s in f.sequence_starts[1:] + [len(text)]:  # across a delimiter, and the final '$'
        qs.append(text[max(0, s - 3):s])
        qs.append(text[s - 1:s])
    return qs + ["#absent", "ZZZZ", "%", "$"]


def check_against_locate(idx, f, queries, mql=None, low_memory=False):
    located = idx.locate(queries, max_query_len=mql, low_memory=low_memory)
    assert sum(len(h) for h in located) > 0
    for P, S_ in PS:
        got = idx.extract(queries, prefix_len=P, suffix_len=S_, max_query_len=mql, low_memory=low_memory)
        assert [r.query_num for r in got] == list(range(len(queries)))
        assert [r.query for r in got] == list(queries)
        want = restate_extract(f.text, f.sequence_starts, f.sequence_names, located, P, S_)
        assert as_rows(got) == want, (P, S_, mql, low_memory)


# ------------------------------------------------------------------ GPU: every golden, every field
@pytest.mark.gpu
@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
@pytest.mark.parametrize("golden", [c[0] for c in GOLDEN_CASES])
def test_extract_matches_restatement_on_goldens(S, golden, low_memory):
    f = parse_sufr((EXPECTED / golden).read_bytes())
    queries = golden_queries(f, golden)
    idx = S.SufrIndex.open(EXPECTED / golden)
    try:
        check_against_locate(idx, f, queries, None, low_memory)
        if golden in ("uniprot-masked.sufr", "long_dna_sequence.sufr", "long_dna_sequence_allow_ambiguity.sufr"):
            for mql in (3, 6):
                check_against_locate(idx, f, queries, mql, low_memory)
    finally:
        idx.close()


@pytest.mark.gpu
def test_extract_on_a_built_index_matches_the_opened_file(S):
    seq = S.read_sequence_file(GOLDEN / "inputs" / "uniprot.fa", b"%")
    f = parse_sufr((EXPECTED / "uniprot.sufr").read_bytes())
    idx, r = device_index(S, seq.seq, seq.start_positions, seq.sequence_names)
    try:
        check_against_locate(idx, f, golden_queries(f, "built"))
        assert idx.string_at(0) == f.text
    finally:
        idx.close()
        r.free()


@pytest.mark.gpu
def test_u64_file_extracts_like_u32(S, tmp_path):
    seq = S.read_sequence_file(GOLDEN / "inputs" / "long_dna_sequence.fa", b"%")
    idxs = []
    for bits in (32, 64):
        path = tmp_path / f"u{bits}.sufr"
        S.SufrBuilder(S.SufrBuilderArgs(text=seq.seq, path=str(path), is_dna=True, sequence_starts=seq.start_positions,
                                        sequence_names=seq.sequence_names), bits)
        idxs.append(S.SufrIndex.open(path))
    a, b = idxs
    try:
        assert b.info["index_bits"] == 64
        queries = ["CATGTTGTCACG", "CCATGGGAC", "ACG", "T", "NNNN", "$"]
        for P, S_ in PS:
            for mql in (None, 6):
                assert as_rows(a.extract(queries, P, S_, mql)) == as_rows(b.extract(queries, P, S_, mql))
        for ln in (None, 0, 17):
            la, lb = a.list(0, None, ln), b.list(0, None, ln)
            assert all(np.array_equal(x, y) for x, y in zip(la[:3], lb[:3])) and la[3] == lb[3]
        assert a.string_at(5, 40) == b.string_at(5, 40) == seq.seq[5:45]
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------ GPU: windows and the byte budget
def concat_windows(idx, total, max_hits, P, S_, max_bytes):
    parts, first = [], 0
    while first < total:
        arrs, data = idx.extract_window(first, min(max_hits, total - first), P, S_, max_bytes=max_bytes)
        assert len(arrs[0]) >= 1  # extract_window retries a region larger than the budget
        assert arrs[4][0] == 0 and int(arrs[4][-1]) == len(data)
        if len(arrs[0]) > 1:
            assert len(data) <= max_bytes
        parts.append((arrs, data))
        first += len(arrs[0])
    cols = [np.concatenate([p[0][k] for p in parts]) for k in range(4)]
    sizes = np.concatenate([np.diff(p[0][4]) for p in parts])
    return cols, sizes, b"".join(p[1] for p in parts)


@pytest.mark.gpu
def test_windows_and_byte_budget(S):
    from sufr_b200 import _lib
    f = parse_sufr((EXPECTED / "long_dna_sequence.sufr").read_bytes())
    idx = S.SufrIndex.open(EXPECTED / "long_dna_sequence.sufr")
    try:
        queries = ["ACG", "TTT", "GA", "CATGTTGTCACG", "ZZZ"]
        _, _, ho = idx.locate_ranges(queries)
        total = int(ho[-1])
        assert total > 50
        for P, S_ in ((3, 5), (0, 0), (10, None)):
            (suf, seq, rs, re_, offs), data = idx.extract_window(0, total, P, S_, max_bytes=1 << 40)
            assert len(suf) == total and int(offs[-1]) == len(data)
            sizes = np.diff(offs)
            assert np.array_equal(sizes, re_ - rs)
            big = int(sizes.sum())
            for mb in sorted({1, 2, 3, 7, 8, 15, 16, 17, 100, big // 3, big - 1, big}):
                if mb < 1:
                    continue
                for mh in (total, total // 3 + 1, 7):
                    cols, sz, d = concat_windows(idx, total, mh, P, S_, mb)
                    assert all(np.array_equal(c, w) for c, w in zip(cols, (suf, seq, rs, re_))), (P, S_, mb, mh)
                    assert np.array_equal(sz, sizes) and d == data, (P, S_, mb, mh)
        # the num == 0 protocol through the C ABI: the first region alone does not fit
        (suf, _, rs, re_, offs), _ = idx.extract_window(0, 4, None, None, max_bytes=1 << 40)
        first_size = int(re_[0] - rs[0])
        assert first_size > 1
        num = C.c_uint64(123)
        bo = np.full(5, 7, np.uint64)
        buf = np.zeros(first_size, np.uint8)
        L = _lib.lib()
        assert L.sufr_b200_index_extract(idx._h, 0, 4, 0, U64_MAX, first_size - 1, C.byref(num), None, None, None, None,
                                         bo.ctypes.data, buf.ctypes.data) == 0
        assert num.value == 0 and bo[0] == 0 and int(bo[1]) == first_size
        assert L.sufr_b200_index_extract(idx._h, 0, 4, 0, U64_MAX, first_size, C.byref(num), None, None, None, None,
                                         bo.ctypes.data, buf.ctypes.data) == 0
        assert num.value >= 1 and int(bo[1]) == first_size
        text, starts, names = f.text, f.sequence_starts, f.sequence_names
        assert buf[:first_size].tobytes() == restate_region(text, starts, int(suf[0]))[4]
        # locate -> extract -> locate (other queries) -> extract: each extract reads the latest locate
        for qs in (["ACGT", "GGG"], ["TTTT", "CATGTTGTCACG", "AAAAA"], ["ACGT"]):
            located = idx.locate(qs)  # (SufrIndex.locate runs sufr_b200_index_locate)
            nh = sum(len(h) for h in located)
            (suf, seq, rs, re_, offs), data = idx.extract_window(0, nh, 2, 4)
            want = [r for rows in restate_extract(text, starts, names, located, 2, 4) for r in rows]
            assert suf.tolist() == [w[1] for w in want]
            assert [(int(a), int(b)) for a, b in zip(rs, re_)] == [w[4] for w in want]
            assert [data[int(offs[i]):int(offs[i + 1])] for i in range(nh)] == [w[6] for w in want]
    finally:
        idx.close()


# ------------------------------------------------------------------ GPU: regions of tens of MB, the end of the text
@pytest.mark.gpu
def test_long_regions_and_the_end_of_the_text(S):
    rng = np.random.default_rng(11)
    lens = [1000, 48_000_003, 17, 5000, 333]
    recs = [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)] for n in lens]
    kmer = np.frombuffer(b"ACGTTGCAACGTTGCAAGGTCA", np.uint8)
    plants = [(0, 10), (1, 100), (1, 23_000_000), (1, lens[1] - len(kmer)), (3, 2500), (4, lens[4] - len(kmer))]
    for r, p in plants:
        recs[r][p:p + len(kmer)] = kmer
    text = b"%".join(r.tobytes() for r in recs) + b"$"
    n = len(text)
    assert n % 16 != 0
    starts = [0]
    for ln in lens[:-1]:
        starts.append(starts[-1] + ln + 1)
    names = [f"r{i}" for i in range(len(lens))]
    idx, res = device_index(S, text, starts, names, is_dna=True)
    try:
        q = kmer.tobytes().decode()
        located = idx.locate([q])
        assert len(located[0]) == len(plants)
        for P, S_ in ((10 ** 9, None), (None, None), (5, None), (10 ** 9, 3)):
            (got,) = as_rows(idx.extract([q], P, S_))
            (want,) = restate_extract(text, starts, names, located, P, S_)
            assert got == want, (P, S_)
            if P == 10 ** 9 and S_ is None:
                assert max(len(x[6]) for x in got) == lens[1] + 1           # the whole 48 Mbp record, delimiter too
                assert any(starts[-1] + len(x[6]) == n for x in got)        # a region that ends at n
        # suffixes that end at n (list with the whole suffix), and short ones of every length near 16
        last = idx.list(res.num_suffixes - 40, 40, None)
        for i in range(40):
            assert last[3][int(last[2][i]):int(last[2][i + 1])] == text[int(last[0][i]):]
        assert idx.string_at(n - 20) == text[-20:]
        assert idx.string_at(n - 1, 100) == b"$"
    finally:
        idx.close()
        res.free()


@pytest.mark.gpu
def test_index_without_sequence_starts(S):
    text = b"ACGTACGTACGTTTGACCA$"
    idx, r = device_index(S, text, (), (), is_dna=True)
    try:
        located = idx.locate(["CGT", "ACC"])
        for P, S_ in PS:
            got = as_rows(idx.extract(["CGT", "ACC"], P, S_))
            assert got == restate_extract(text, [], [], located, P, S_)
            assert all(x[2] is None and x[3] == 0 for rows in got for x in rows)
        (rows,) = as_rows(idx.extract(["CGT"], 1000, None))
        assert all(x[4] == (0, len(text)) and x[6] == text for x in rows)
    finally:
        idx.close()
        r.free()


# ------------------------------------------------------------------ GPU: list and string_at
@pytest.mark.gpu
@pytest.mark.parametrize("golden", ["2.sufr", "abba.sufr", "long_dna_sequence.sufr", "uniprot.sufr",
                                    "uniprot-masked.sufr"])
def test_list_matches_the_file(S, golden):
    f = parse_sufr((EXPECTED / golden).read_bytes())
    s, n = f.num_suffixes, f.text_len
    idx = S.SufrIndex.open(EXPECTED / golden)
    rng = random.Random(golden)
    try:
        windows = [(0, s), (0, 1), (s - 1, 1), (s - 1, None), (s, 0), (3, 0)]
        windows += [(a, rng.randrange(0, s - a + 1)) for a in (rng.randrange(s) for _ in range(6))]
        for ln in (None, 0, 1, 7, 16, 17):
            for first, count in windows:
                suf, lcp, offs, data = idx.list(first, count, ln)
                cnt = s - first if count is None else count
                assert np.array_equal(suf, f.sa[first:first + cnt].astype(np.uint64))
                assert np.array_equal(lcp, f.lcp[first:first + cnt].astype(np.uint64))
                want = [f.text[p:n if ln is None else min(p + ln, n)] for p in suf.tolist()]
                assert len(offs) == cnt + 1 and offs[0] == 0
                assert [data[int(offs[i]):int(offs[i + 1])] for i in range(cnt)] == want, (ln, first, count)
        # small windows and budgets: the same rows
        whole = idx.list(0, None, 17)
        small = idx.list(0, None, 17, rows_window=5, max_bytes=20)
        assert all(np.array_equal(x, y) for x, y in zip(whole[:3], small[:3])) and whole[3] == small[3]
        # string_at
        assert idx.string_at(0) == f.text
        assert idx.string_at(0, 1) == f.text[:1]
        assert idx.string_at(n - 1) == f.text[-1:]
        assert idx.string_at(n) == b"" and idx.string_at(n, 5) == b""
        assert idx.string_at(n - 3, 10 ** 12) == f.text[-3:]
        assert idx.string_at(2, 0) == b""
        for p in sorted({1, n // 2, max(0, n - 17)}):  # (abba.sufr: n = 15)
            for ln in (1, 15, 16, 17, None):
                assert idx.string_at(p, ln) == f.text[p:n if ln is None else p + ln]
    finally:
        idx.close()


# ------------------------------------------------------------------ GPU: argument errors
@pytest.mark.gpu
def test_argument_errors_leave_the_index_usable(S):
    from sufr_b200 import _lib
    f = parse_sufr((EXPECTED / "2.sufr").read_bytes())
    idx = S.SufrIndex.open(EXPECTED / "2.sufr")
    L = _lib.lib()
    try:
        def refused(fn):
            with pytest.raises(S.SufrError) as e:
                fn()
            assert e.value.code == _lib.ERR_ARGUMENT

        refused(lambda: idx.extract_window(0, 1))  # no locate yet
        located = idx.locate(["GT"])
        refused(lambda: idx.extract_window(0, 5))
        refused(lambda: idx.extract_window(5, 0))
        refused(lambda: idx.extract_window(3, 2))
        refused(lambda: idx.list(f.num_suffixes + 1, 0))
        refused(lambda: idx.list(f.num_suffixes - 1, 2))
        refused(lambda: idx.string_at(f.text_len + 1))
        refused(lambda: idx.string_at(-2))
        refused(lambda: idx.list(-1, 1))
        refused(lambda: idx.extract_window(-1, 1))
        num = C.c_uint64()
        bo = np.zeros(3, np.uint64)
        buf = np.zeros(64, np.uint8)
        assert L.sufr_b200_index_extract(idx._h, 0, 2, 0, 0, 64, C.byref(num), None, None, None, None, None,
                                         buf.ctypes.data) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_extract(idx._h, 0, 2, 0, 0, 64, C.byref(num), None, None, None, None, bo.ctypes.data,
                                         None) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_extract(idx._h, 0, 2, 0, 0, 64, None, None, None, None, None, bo.ctypes.data,
                                         buf.ctypes.data) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_list(idx._h, 0, 2, 4, 64, C.byref(num), None, None, None,
                                      buf.ctypes.data) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_list(idx._h, 0, 2, 4, 64, C.byref(num), None, None, bo.ctypes.data,
                                      None) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_string_at(idx._h, 0, 4, buf.ctypes.data, None) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_string_at(idx._h, 0, 4, None, C.byref(num)) == _lib.ERR_ARGUMENT
        assert L.sufr_b200_index_extract(None, 0, 0, 0, 0, 0, C.byref(num), None, None, None, None, bo.ctypes.data,
                                         buf.ctypes.data) == _lib.ERR_ARGUMENT
        # still answers
        assert idx.locate(["GT"]) == located
        (rows,) = as_rows(idx.extract(["GT"], 1, 2))
        assert [(x[1], x[2], x[4], x[6]) for x in rows] == [(15, "DEF", (5, 8), b"CGT"), (6, "ABC", (5, 8), b"CGT"),
                                                           (11, "DEF", (1, 4), b"CGT"), (2, "ABC", (1, 4), b"CGT")]
        (rows,) = as_rows(idx.extract(["GT"], 1, None))
        assert [x[6] for x in rows[:2]] == [b"CGT$", b"CGT%"]
        assert idx.string_at(9, 4) == b"ACGT"
    finally:
        idx.close()
