"""k-mer counting on a device index (sufr_b200_index_kmer_spectrum / _kmers / _kmer_multiplicity, SufrIndex.kmer_spectrum
/ .kmers / .kmer_multiplicity) against the host reference of tests/kmer_reference.py, which reads the text alone.

CPU tests tie the reference to a hand-worked table and to the groups of the spec sorter's suffix / LCP arrays.  GPU
tests compare every field over device builds and reopened files (u32 and u64), plain / DNA / ambiguity indexes, build
caps 5 and 32, every golden file, texts of 1 to 17 bytes, and a 16 M DNA text with planted repeats."""
import ctypes as C
import random

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES
from index_matrix import ACGT, ALL, PROTEIN, IndexMatrix, make_text, with_records
import kmer_reference as K

EXPECTED = GOLDEN / "expected"
U64_MAX = 0xFFFFFFFFFFFFFFFF

# ------------------------------------------------------------------ CPU: the reference itself
# (text, starts, is_dna, k) -> {k-mer: count}
HAND = [
    (b"BANANA", [], False, 1, {b"A": 2, b"B": 1, b"N": 2}),       # the last byte is the record's own
    (b"BANANA", [], False, 2, {b"AN": 2, b"BA": 1, b"NA": 1}),
    (b"BANANA", [], False, 5, {b"BANAN": 1}),                       # ends at the last byte a k-mer may hold
    (b"BANANA", [], False, 6, {}),
    # two DNA records: ACGNAC% and ACA$; N breaks k-mers, '%' and '$' are the records' last bytes
    (b"ACGNAC%ACA$", [0, 7], True, 2, {b"AC": 3, b"CG": 1, b"CA": 1}),
    (b"ACGNAC%ACA$", [0, 7], True, 3, {b"ACG": 1, b"ACA": 1}),
    (b"ACGNAC%ACA$", [0, 7], True, 4, {}),                          # longer than both records allow
    (b"ACGNAC%ACA$", [0, 7], False, 3, {b"ACG": 1, b"CGN": 1, b"GNA": 1, b"NAC": 1, b"ACA": 1}),
    (b"xACG%", [1], True, 2, {b"AC": 1, b"CG": 1}),                 # [0, 1) before the first start: its byte is its last
]


@pytest.mark.parametrize("row", range(len(HAND)))
def test_reference_hand_worked(row):
    text, starts, dna, k, want = HAND[row]
    assert dict(K.counts(text, k, starts, dna)) == want
    keys, cnt = K.distinct(text, k, starts, dna)
    assert keys == sorted(want) and cnt == [want[x] for x in keys]
    h, d, o, m = K.spectrum(text, k, starts, dna, 3)
    assert d == len(want) and o == sum(want.values()) and m == max(want.values(), default=0)
    mult = K.multiplicity(text, k, starts, dna)
    assert int((mult.astype(np.int64)).sum()) == sum(v * v for v in want.values())


def test_reference_against_spec_groups():
    """On small random texts the groups of the spec sorter's arrays (LCP < k) are the reference's distinct k-mers."""
    import oracle as O
    rng = random.Random(5)
    for trial in range(30):
        dna = trial % 2 == 0
        alpha = b"ACGTN" if dna else b"AB%"
        n = rng.randrange(1, 40)
        text = bytes(rng.choice(alpha) for _ in range(n)) + b"$"
        starts = [0] + sorted(rng.sample(range(1, n + 1), min(n, rng.randrange(0, 3))))
        t, sa, lcp = O.spec_build(text, is_dna=dna, allow_ambiguity=dna and trial % 4 == 0)
        for k in (1, 2, 3, 5):
            occ = set(K.occurrences(t, k, starts, dna).tolist())
            assert occ <= set(sa)  # every occurrence is an indexed position
            groups = [g for g in K.groups_from_arrays(sa, lcp, k, occ) if g[2]]
            keys, cnt = K.distinct(t, k, starts, dna)
            assert [t[g[3]:g[3] + k] for g in groups] == keys, (text, k)
            assert [g[2] for g in groups] == cnt


# ------------------------------------------------------------------ GPU fixtures
def n_run_text():
    t = bytearray(make_text(50, 6000, ACGT, copies=60, runs=[(b"T", 40)], rare=b"N", rare_p=0.01))
    t[2000:3200] = b"N" * 1200  # an N run of 1200: the N-run LCP rule
    return bytes(t)


SPECS = {
    "plain_acgt": (with_records(make_text(61, 4000, ACGT, copies=40, runs=[(b"T", 40)]), 8, 1), dict(), ALL),
    "dna_N": (with_records(make_text(62, 4000, ACGT, copies=40, runs=[(b"A", 30)], rare=b"N", rare_p=0.01), 8, 2),
              dict(is_dna=True), ALL),
    "dna_amb_Nrun": (with_records(n_run_text(), 6, 3), dict(is_dna=True, allow_ambiguity=True), ALL),
    "protein_q5": (with_records(make_text(64, 5000, PROTEIN, copies=80), 6, 4), dict(max_query_len=5), ALL),
    "dna_q32": (with_records(make_text(65, 6000, ACGT, copies=60, copy_len=(30, 200), runs=[(b"AC", 50)]), 6, 5),
                dict(is_dna=True, max_query_len=32), [("built", 32), ("file", 64)]),
    "plain_delim_inside": ((b"AB%AB%AB%ABAB$", [0, 3, 9], ["r0", "r1", "r2"]), dict(), ALL),
}
for _n in (1, 2, 3, 5, 8, 13, 17):  # tiny texts: windows that end at n and at s
    SPECS[f"tiny_{_n}"] = ((bytes(random.Random(_n).choice(b"AC") for _ in range(_n - 1)) + b"$", [0], ["r0"]),
                           dict(is_dna=True), [("built", 32), ("file", 64)])


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


class Case(IndexMatrix):
    def __init__(self, S, name, tmp):
        (text, starts, names), flags, sources = SPECS[name]
        super().__init__(S, name, text, starts, names, flags, sources, tmp)
        self.text = text
        self.dna = bool(flags.get("is_dna"))
        self.cap = flags.get("max_query_len") or 0

    def ks(self):
        n = len(self.text)
        cuts = sorted(set(self.starts) | {n})
        longest = max([b - a for a, b in zip([0] + cuts, cuts)] or [1])
        ks = {1, 2, 21, 31, longest, n + 1}
        if self.cap:
            ks = {k for k in ks if k <= self.cap} | {self.cap}
        return sorted(ks)


@pytest.fixture(scope="module", params=list(SPECS))
def case(request, S, tmp_path_factory):
    c = Case(S, request.param, tmp_path_factory.mktemp("kmers"))
    yield c
    c.close()


def check_index(S, index, text, starts, dna, k, cap=0):
    """Every field of the three calls against the reference, for one k."""
    keys, cnt = K.distinct(text, k, starts, dna)
    top = max(cnt, default=0)
    for nb in sorted({1, 2, top + 1, 10000}):
        h, d, o, m = K.spectrum(text, k, starts, dna, nb)
        got = index.kmer_spectrum(k, nb)
        assert np.array_equal(got.histogram, h), (k, nb)
        assert (got.distinct, got.occurrences, got.max_count) == (d, o, m), (k, nb)
        assert int(got.histogram.sum()) == got.distinct
        if nb > top:
            assert sum((i + 1) * int(x) for i, x in enumerate(got.histogram)) == got.occurrences
    rb, re_, c, km = index.kmers(k)
    assert [bytes(x) for x in km] == keys, k
    assert c.tolist() == cnt
    if keys:
        ranges = index.search(keys[:200])
        assert ranges == list(zip(rb[:200].tolist(), re_[:200].tolist())), k
    for w in (1, 7, 4096):
        wb, we, wc, wk = index.kmers(k, window=w)
        assert np.array_equal(wb, rb) and np.array_equal(we, re_) and np.array_equal(wc, c) and np.array_equal(wk, km)
    for lo, hi in ((2, None), (1, 1), (3, 5)):
        fb, _, fc, fk = index.kmers(k, min_count=lo, max_count=hi)
        sel = [i for i, x in enumerate(cnt) if x >= lo and (hi is None or x <= hi)]
        assert [bytes(x) for x in fk] == [keys[i] for i in sel] and fc.tolist() == [cnt[i] for i in sel]
    want = K.multiplicity(text, k, starts, dna)
    got = index.kmer_multiplicity(k)
    assert np.array_equal(got, want), k
    assert int(got.astype(np.int64).sum()) == sum(x * x for x in cnt)
    n = len(text)
    for a, ln in ((0, min(n, 5)), (n // 2, min(n - n // 2, 9)), (max(0, n - 7), min(n, 7)), (n, 0)):
        assert np.array_equal(index.kmer_multiplicity(k, a, ln), want[a:a + ln]), (k, a, ln)
    assert np.array_equal(index.kmer_multiplicity(k, window=3), want)


@pytest.mark.gpu
def test_kmers_match_reference(case, S):
    for label, index in case.indexes:
        for k in case.ks():
            check_index(S, index, case.text, case.starts, case.dna, k, case.cap)


@pytest.mark.gpu
def test_kmers_cap_refused_and_state_untouched(case, S):
    L = S._lib.lib()
    q = [case.text[:3], case.text[-4:-1]]
    for label, index in case.indexes:
        _, _, ho = index.locate_ranges(q)
        before = [x.tolist() for x in index.hits(0, int(ho[-1]))]
        if case.cap:
            with pytest.raises(S.SufrError) as e:
                index.kmer_spectrum(case.cap + 1)
            assert e.value.code == S._lib.ERR_ARGUMENT
        num, nxt = C.c_uint64(), C.c_uint64()
        h = np.zeros(4, np.uint64)
        u = np.zeros(4, np.uint64)
        s = index._s
        bad = [
            lambda: L.sufr_b200_index_kmer_spectrum(index._h, 0, 4, h.ctypes.data, None, None, None),
            lambda: L.sufr_b200_index_kmer_spectrum(index._h, 1, 0, h.ctypes.data, None, None, None),
            lambda: L.sufr_b200_index_kmer_spectrum(index._h, 1, 65537, h.ctypes.data, None, None, None),
            lambda: L.sufr_b200_index_kmer_spectrum(index._h, 1, 4, None, None, None, None),
            lambda: L.sufr_b200_index_kmers(index._h, 1, 3, 2, 0, 4, C.byref(num), C.byref(nxt), u.ctypes.data,
                                            u.ctypes.data, u.ctypes.data, None),
            lambda: L.sufr_b200_index_kmers(index._h, 1, 1, U64_MAX, s + 1, 4, C.byref(num), C.byref(nxt),
                                            u.ctypes.data, u.ctypes.data, u.ctypes.data, None),
            lambda: L.sufr_b200_index_kmer_multiplicity(index._h, 1, len(case.text), 1, h.ctypes.data),
            lambda: L.sufr_b200_index_kmer_multiplicity(index._h, 1, 0, len(case.text) + 1, h.ctypes.data),
        ]
        for f in bad:
            assert f() == S._lib.ERR_ARGUMENT
        for f in (lambda: index.kmer_spectrum(-1), lambda: index.kmers(0), lambda: index.kmer_multiplicity(1, -1)):
            with pytest.raises(S.SufrError):
                f()
        check_index(S, index, case.text, case.starts, case.dna, 2)
        assert [x.tolist() for x in index.hits(0, int(ho[-1]))] == before  # the locate state is the one before


@pytest.mark.gpu
def test_kmers_window_from_inside_a_group(case, S):
    """first_rank inside a group lists from the next group that starts at or after it; max_kmers = 1 steps one
    group at a time."""
    L = S._lib.lib()
    index = case.indexes[0][1]
    rb, re_, c, _ = index.kmers(2)
    num, nxt = C.c_uint64(), C.c_uint64()
    out = [np.zeros(4, np.uint64) for _ in range(3)]
    for b, e in zip(rb.tolist(), re_.tolist()):
        if e - b < 2:
            continue
        assert L.sufr_b200_index_kmers(index._h, 2, 1, U64_MAX, b + 1, 4, C.byref(num), C.byref(nxt),
                                       *[o.ctypes.data for o in out], None) == 0
        later = [i for i, x in enumerate(rb.tolist()) if x >= b + 1][:4]
        assert out[0][:num.value].tolist() == [int(rb[i]) for i in later]
        break
    first, seen = 0, []
    while first < index._s:
        assert L.sufr_b200_index_kmers(index._h, 2, 1, U64_MAX, first, 1, C.byref(num), C.byref(nxt),
                                       *[o.ctypes.data for o in out], None) == 0
        assert num.value <= 1 and nxt.value > first
        seen += out[0][:num.value].tolist()
        first = nxt.value
    assert seen == rb.tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("golden", [g for g, _, _ in GOLDEN_CASES])
def test_kmers_golden(golden, S):
    index = S.SufrIndex.open(EXPECTED / golden)
    try:
        info = index.info
        if info["seed_mask"] is not None:
            for f in (lambda: index.kmer_spectrum(2), lambda: index.kmers(2), lambda: index.kmer_multiplicity(2)):
                with pytest.raises(S.SufrError) as e:
                    f()
                assert e.value.code == S._lib.ERR_UNSUPPORTED
            return
        text = index.string_at(0)
        cap = info["max_query_len"] or 0
        for k in (1, 2, 5, 21):
            if cap and k > cap:
                continue
            check_index(S, index, text, info["sequence_starts"], bool(info["is_dna"]), k, cap)
    finally:
        index.close()


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [32, 64])
def test_kmers_16M_planted_repeats(bits, S):
    """A 16 M DNA text with planted repeats and N, checked in numpy from the text (2-bit k-mer codes)."""
    import torch
    rng = np.random.default_rng(11)
    n = 1 << 24
    t = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    for _ in range(2000):  # planted repeats
        a, b, ln = rng.integers(0, n - 5000, 2).tolist() + [int(rng.integers(21, 3000))]
        t[b:b + ln] = t[a:a + ln]
    t[rng.integers(0, n, 3000)] = ord("N")
    t[-1] = ord("$")
    starts = [0, n // 3, 2 * n // 3]
    for c in starts[1:]:
        t[c - 1] = ord("%")
    text = t.tobytes()
    dt = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", is_dna=True, sequence_starts=starts, sequence_names=["a", "b", "c"])
    r = S.build(args, index_bits=bits, result_memory=S.MEM_DEVICE, device_text=(dt.data_ptr(), dt.numel()))
    index = S.SufrIndex(r, args)
    try:
        for k in (21, 31):
            occ = K.occurrences(text, k, starts, True)
            code = np.zeros(len(occ), np.int64)
            lut = np.zeros(256, np.int64)
            lut[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4)
            for j in range(k):
                code = code * 4 + lut[t[occ + j]]
            keys, inv, cnt = np.unique(code, return_inverse=True, return_counts=True)
            sp = index.kmer_spectrum(k, 100)
            want_h = np.bincount(np.minimum(cnt, 100) - 1, minlength=100).astype(np.uint64)
            assert np.array_equal(sp.histogram, want_h)
            assert (sp.distinct, sp.occurrences, sp.max_count) == (len(keys), len(occ), int(cnt.max()))
            rb, re_, c, km = index.kmers(k, min_count=2, window=1 << 16)
            sel = cnt >= 2
            assert np.array_equal(c, cnt[sel].astype(np.uint64))
            got_code = np.zeros(len(km), np.int64)
            for j in range(k):
                got_code = got_code * 4 + lut[km[:, j]]
            assert np.array_equal(got_code, keys[sel])
            mult = np.zeros(n, np.uint32)
            mult[occ] = cnt[inv]
            assert np.array_equal(index.kmer_multiplicity(k, window=1 << 22), mult)
    finally:
        index.close()
        r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [32, 64])
def test_kmers_group_longer_than_chunk(bits, S):
    """A poly-A run makes one group of about 200 000 ranks, more than an enumeration chunk of a small window: the
    window that starts at it lists it whole, and every window size gives the same k-mers."""
    import torch
    text = b"ACGT" * 50 + b"A" * 200_000 + b"CAGT" * 30 + b"$"
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", is_dna=True)
    r = S.build(args, index_bits=bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    index = S.SufrIndex(r, args)
    try:
        for k in (2, 21):
            keys, cnt = K.distinct(text, k, [], True)
            for w in (1, 3, 1 << 24):
                rb, re_, c, km = index.kmers(k, window=w)
                assert [bytes(x) for x in km] == keys and c.tolist() == cnt, (k, w)
                assert index.search(keys) == list(zip(rb.tolist(), re_.tolist()))
            fb, _, fc, _ = index.kmers(k, min_count=1000, window=1)
            assert fc.tolist() == [x for x in cnt if x >= 1000]
            assert np.array_equal(index.kmer_multiplicity(k, window=1 << 16), K.multiplicity(text, k, [], True))
    finally:
        index.close()
        r.free()
