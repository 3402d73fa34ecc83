"""The GPU search (`search_kernel`: compare, search_first / search_last, the rank mapping of the LCP-subsampled array)
against a host reference of the match set (tests/search_reference.py), query by query, over every index mode.

CPU tests tie the reference to the reference implementation's own query fixtures (from the golden `.sufr` files
alone) and to a hand-worked table.  GPU tests compare `search` in both memory modes, `count` and `locate_ranges` for
EVERY query of a matrix of index sources (device build, written and reopened file; u32 and u64), index modes (plain,
DNA, DNA with ambiguity, build caps, seed masks), alphabets, sizes (1 suffix to 2 M) and run-time caps."""
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
import search_reference as R
from sufrfile import parse_sufr
from test_file_query import CLI_FIXTURES, _want, format_locate

EXPECTED = GOLDEN / "expected"
EXE = ROOT / "sufr_b200" / "sufr-b200"
NONE = 0xFFFFFFFFFFFFFFFF


def file_index(path) -> R.Index:
    f = parse_sufr(Path(path).read_bytes())
    return R.Index(f.text, f.sa, f.lcp, 0 if f.seed_mask else f.max_query_len, f.seed_mask)


# ------------------------------------------------------------------ CPU: the reference itself
def _hits(f, ranges):
    """SufrFile::locate's hits (rank, suffix, name, position) of rank ranges over a parsed file."""
    starts = np.asarray(f.sequence_starts, dtype=np.int64)
    out = []
    for r in ranges:
        hs = []
        if r is not None:
            for rank in range(*r):
                suf = int(f.sa[rank])
                k = int(np.searchsorted(starts, suf, side="right")) - 1
                hs.append((rank, suf, f.sequence_names[k], suf - int(starts[k])))
        out.append(hs)
    return out


@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
@pytest.mark.parametrize("case", CLI_FIXTURES, ids=[c[0] for c in CLI_FIXTURES])
def test_reference_reproduces_query_fixtures(case, low_memory):
    """From the golden files alone, the match sets give the reference implementation's locate outputs, seed mask and
    run-time -m 3 / -m 6 included."""
    fixture, sufr, flags, queries = case
    mql = int(flags[1]) if flags[:1] == ["-m"] else None
    f = parse_sufr((EXPECTED / sufr).read_bytes())
    idx = R.Index(f.text, f.sa, f.lcp, 0 if f.seed_mask else f.max_query_len, f.seed_mask)
    got = R.expected(idx, [q.encode() for q in queries], mql, low_memory)
    assert format_locate(queries, _hits(f, got), "-a" in flags) == _want(fixture)


# The last m-prefix group of a golden file, searched in memory with a run-time cap m: one sampled entry matches and it
# is the last one, so the range ends at the number of suffixes.
LAST_SAMPLED = [
    # (file, m, query, full-array range, true matches)
    ("long_dna_sequence.sufr", 6, b"TTTTTT", (19997, 20001), 4),
    ("long_dna_sequence.sufr", 3, b"TTT", (19682, 20001), 319),
    ("3.sufr", 6, b"TTTTCA", (100, 101), 1),
    ("uniprot.sufr", 6, b"YYYYQE", (63219, 63220), 1),
]


@pytest.mark.parametrize("case", LAST_SAMPLED, ids=[f"{c[0]}-m{c[1]}" for c in LAST_SAMPLED])
def test_reference_last_sampled_goldens(case):
    name, m, q, full, true = case
    idx = file_index(EXPECTED / name)
    assert full[1] == idx.s and full[1] - full[0] == true
    assert R.full_ranges(idx, [q], m) == [full]
    assert R.expected(idx, [q], m, low_memory=True) == [full]
    sampled = np.flatnonzero(idx.lcp < m)
    assert sampled[-1] == full[0]  # the last sampled entry
    assert R.expected(idx, [q], m, low_memory=False) == [full]


# Hand-worked indexes: (text, SA, LCP, build cap, seed mask) and (query, run-time cap, full range, in-memory range).
HAND = {
    # capped, Q = 2: keys AB {0, 2, 4} and BA {1, 3} tie, in position-descending order, with LCP exactly Q
    "capped": ((b"ABABAB", [4, 2, 0, 5, 3, 1], [0, 2, 2, 0, 1, 2], 2, None), [
        (b"AB", None, (0, 3), (0, 3)),
        (b"ABA", None, (0, 3), (0, 3)),      # compared on the first Q bytes only
        (b"ABBB", 0, (0, 3), (0, 3)),        # a run-time cap of 0 is no cap
        (b"B", None, (3, 6), (3, 6)),
        (b"BAB", 1, (3, 6), (3, 6)),         # sampled {0, 3}: 3 is the last one, so the end is s = 6
        (b"A", 1, (0, 3), (0, 3)),           # one sampled entry: the end is the next sampled rank
        (b"", 1, (0, 6), (0, 4)),            # two sampled entries: the last sampled rank + 1
        (b"", None, (0, 6), (0, 6)),
        (b"C", None, None, None),
        (b"BB", 5, None, None),
    ]),
    # seed mask 101 (care offsets 0 and 2): keys AC {1, 4}, C (6), CG (3), CT (0), G (5), TA (2); LCP in care units
    "mask": ((b"CATCAGC", [4, 1, 6, 3, 0, 5, 2], [0, 2, 0, 1, 1, 0, 0], 0, "101"), [
        (b"AGC", None, (0, 2), (0, 2)),      # the byte under the 0 is not compared
        (b"C", None, (2, 5), (2, 5)),
        (b"CXG", None, (3, 4), (3, 4)),
        (b"CXT", 1, (2, 5), (2, 5)),         # sampled {0, 2, 5, 6}: one in the range, the next one ends it
        (b"T", 1, (6, 7), (6, 7)),           # the last sampled entry: the end is s = 7
        (b"GXA", None, None, None),          # care offset 2 runs past the end of the text
        (b"G", 0, (5, 6), (5, 6)),
        (b"", 1, (0, 7), (0, 7)),
    ]),
    # uncapped: the suffix array of BANANA (no sentinel)
    "last_sampled": ((b"BANANA", [5, 3, 1, 0, 4, 2], [0, 1, 3, 0, 0, 2], 0, None), [
        (b"NA", 1, (4, 6), (4, 6)),          # sampled {0, 3, 4}: 4 is the last one, so the end is s = 6
        (b"NAN", 2, (4, 6), (4, 6)),         # sampled {0, 1, 3, 4}
        (b"A", 1, (0, 3), (0, 3)),
        (b"ANA", 2, (1, 3), (1, 3)),
        (b"", 2, (0, 6), (0, 5)),
        (b"BANANA", None, (3, 4), (3, 4)),
        (b"BANANAS", None, None, None),      # runs past the end of the text
        (b"NANA", None, (5, 6), (5, 6)),
        (b"A", None, (0, 3), (0, 3)),
    ]),
}


@pytest.mark.parametrize("name", list(HAND))
def test_reference_hand_worked(name):
    import oracle as O
    (text, sa, lcp, cap, mask), rows = HAND[name]
    _, spec_sa, spec_lcp = O.spec_build(text, max_query_len=cap or None, seed_mask_str=mask)
    assert (spec_sa, spec_lcp) == (sa, lcp)  # the table's arrays are those of the index definition
    idx = R.Index(text, np.array(sa), np.array(lcp), cap, mask)
    for q, m, full, mem in rows:
        assert R.full_ranges(idx, [q], m) == [full], (q, m)
        assert R.expected(idx, [q], m, low_memory=True) == [full], (q, m)
        assert R.expected(idx, [q], m, low_memory=False) == [mem], (q, m)


def test_reference_against_brute_force():
    """The vectorised matcher (positions sorted by their first 8 compared bytes, the bytes beyond compared one by one)
    against a scan of every suffix."""
    rng = random.Random(5)
    text = bytes(rng.choice(b"AC") for _ in range(300)) + b"AAAAAAAAAAAAAAAAAAAAAAAA"
    sa = sorted(range(len(text)), key=lambda p: text[p:])
    idx = R.Index(text, np.array(sa), np.zeros(len(sa), np.int64))
    qs = [text[p:p + ln] for p in range(0, len(text), 7) for ln in (1, 5, 8, 9, 15, 30)] + [b"A" * 20, b"A" * 25]
    for q, got in zip(qs, R.full_ranges(idx, qs)):
        ranks = sorted(i for i, p in enumerate(sa) if text[p:p + len(q)] == q)
        assert got == ((ranks[0], ranks[-1] + 1) if ranks else None), q
    mask = "111010010100110111"  # 11 care offsets: 8 in the key, 3 beyond
    key = (lambda p: bytes(text[p + o] for o in R.mask_positions(mask) if p + o < len(text)))
    msa = sorted(range(len(text)), key=lambda p: (key(p), -p))
    midx = R.Index(text, np.array(msa), np.zeros(len(msa), np.int64), 0, mask)
    qs = [text[p:p + ln] for p in range(0, len(text), 5) for ln in (1, 2, 3, 5, 12, 14, 18)]
    for q, got in zip(qs, R.full_ranges(midx, qs)):
        c = [o for o in R.mask_positions(mask) if o < len(q)]
        ranks = [i for i, p in enumerate(msa) if all(p + o < len(text) and text[p + o] == q[o] for o in c)]
        assert got == ((ranks[0], ranks[-1] + 1) if ranks else None), q


# ------------------------------------------------------------------ GPU: search_kernel against the reference
def make_text(seed, n, alphabet, *, copies=0, copy_len=(10, 100), runs=(), rare=b"", rare_p=0.0, dollar=True):
    """n random bytes of `alphabet`, with `copies` segments copied from elsewhere in the text (repeats, long LCPs),
    tandem runs of the given units, and bytes of `rare` sprinkled at rate rare_p."""
    rng = np.random.default_rng(seed)
    t = np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)]
    for _ in range(copies):
        ln = int(rng.integers(copy_len[0], copy_len[1] + 1))
        if ln >= n:
            continue
        src, dst = (int(x) for x in rng.integers(0, n - ln, 2))
        t[dst:dst + ln] = t[src:src + ln].copy()
    for unit, count in runs:
        u = np.frombuffer(unit, np.uint8)
        ln = min(n, len(u) * count)
        dst = int(rng.integers(0, n - ln + 1))
        t[dst:dst + ln] = np.tile(u, count)[:ln]
    if rare:
        hit = np.flatnonzero(rng.random(n) < rare_p)
        t[hit] = np.frombuffer(rare, np.uint8)[rng.integers(0, len(rare), len(hit))]
    return t.tobytes() + (b"$" if dollar else b"")


ACGT, PROTEIN = b"ACGT", b"ACDEFGHIKLMNPQRSTVWY"
WIDE = bytes(range(1, 97)) + bytes(range(123, 256))  # (lowercase bytes would be uppercased by the build)
ALL = [("built", 32), ("built", 64), ("file", 32), ("file", 64)]
MASKS = ["101", "11011", "10111011", "1101101101", "111010010100110111"]

# name -> (text, build flags, index sources, query generator settings)
SPECS = {
    "tiny_1": (b"NNNA", dict(is_dna=True), ALL),
    "tiny_2": (b"NNA$", dict(is_dna=True), ALL),
    "tiny_3": (b"NAC$", dict(is_dna=True), ALL),
    "tiny_3_q2": (b"NAAA", dict(is_dna=True, max_query_len=2), ALL),
    "tiny_2_mask": (b"NNAC", dict(is_dna=True, seed_mask="101"), ALL),
    "acgt_plain_4k": (make_text(1, 4000, ACGT, copies=40, runs=[(b"T", 40)]), dict(), ALL),
    "dna_N_4k": (make_text(2, 4000, ACGT, copies=40, runs=[(b"T", 30)], rare=b"N%", rare_p=0.01), dict(is_dna=True), ALL),
    "dna_N_amb_4k": (make_text(2, 4000, ACGT, copies=40, runs=[(b"T", 30)], rare=b"N%", rare_p=0.01),
                     dict(is_dna=True, allow_ambiguity=True), ALL),
    "protein_q5": (make_text(3, 5000, PROTEIN, copies=80), dict(max_query_len=5), ALL),
    "protein_q12_nodollar": (make_text(4, 5000, PROTEIN, copies=80, dollar=False), dict(max_query_len=12), ALL),
    "dna_q32": (make_text(5, 6000, ACGT, copies=60, copy_len=(30, 200), runs=[(b"AC", 50)]),
                dict(is_dna=True, max_query_len=32), ALL),
    "wide_nodollar": (make_text(6, 3000, WIDE, copies=30, dollar=False), dict(), ALL),
    "dna_200k": (make_text(7, 200_000, ACGT, copies=200, copy_len=(20, 2000), runs=[(b"T", 200), (b"ACG", 100)],
                           rare=b"N", rare_p=0.0005), dict(is_dna=True), [("built", 32), ("file", 64)]),
    "protein_200k_q12": (make_text(8, 200_000, PROTEIN, copies=400, copy_len=(12, 300)), dict(max_query_len=12),
                         [("built", 32), ("file", 32)]),
    "dna_2M": (make_text(9, 2_000_000, ACGT, copies=300, copy_len=(1000, 20000), runs=[(b"T", 3000)]),
               dict(is_dna=True), [("built", 32), ("file", 64)]),
}
for _i, _m in enumerate(MASKS):
    _alpha = PROTEIN if _m == "10111011" else ACGT
    SPECS[f"mask_{_m}"] = (make_text(20 + _i, 4000, _alpha, copies=40, rare=b"N" if _alpha == ACGT else b"",
                                     rare_p=0.005, dollar=_i % 2 == 0),
                           dict(is_dna=_alpha == ACGT, seed_mask=_m), ALL)
SPECS["mask_11011_200k"] = (make_text(30, 200_000, ACGT, copies=200, copy_len=(20, 2000)),
                            dict(is_dna=True, seed_mask="11011"), [("built", 32), ("file", 64)])


def run_caps(flags, n):
    caps = [None, 0, 1, 3, 6]
    if flags.get("seed_mask"):
        w = len(R.mask_positions(flags["seed_mask"]))
        caps += [w - 1, w, w + 1, w + 5]
    elif flags.get("max_query_len"):
        q = flags["max_query_len"]
        caps += [q - 1, q, q + 5]
    else:
        caps += [12, 32, n + 1]
    return list(dict.fromkeys(c for c in caps if c is None or c >= 0))


def make_queries(idx: R.Index, seed, caps, alphabet):
    """Every kind of query of the issue list, as bytes."""
    rng = random.Random(seed)
    t, n, sa = idx.text, idx.n, idx.sa
    cap = idx.build_mql or (len(idx.seed_mask) if idx.seed_mask else 24)
    longest = cap + 8
    qs = []
    # substrings at random positions, of lengths 1 to past the cap / mask length
    count = 300 if n < 10 else min(4000, 2 * n)
    for _ in range(count):
        p = rng.randrange(n)
        qs.append(t[p:p + rng.randrange(1, longest + 1)])
    # for every k, the smallest and the largest k-prefix present (the first and last ranks), and the prefix of the last
    # sampled suffix of every subsample a run-time cap selects
    lens = n - sa
    for k in range(1, 13):
        ok = np.flatnonzero(lens >= k)
        if len(ok):
            for r in (ok[0], ok[-1]):
                qs.append(t[sa[r]:sa[r] + k])
    for m in caps:
        if m:
            r = np.flatnonzero(idx.lcp < m)
            if len(r):
                p = int(sa[r[-1]])
                qs += [t[p:p + m], t[p:p + m + 3], t[p:p + len(idx.seed_mask or "") + 2]]
    # prefixes of the first and last suffixes in the suffix array
    for r in (0, len(sa) - 1):
        p = int(sa[r])
        qs += [t[p:p + k] for k in range(1, min(n - p, longest) + 1)]
    # random strings, mostly absent
    qs += [bytes(rng.choice(alphabet) for _ in range(rng.randrange(1, longest + 1))) for _ in range(min(count, 500))]
    # bytes the text does not have
    qs += [b"\x01", b"\xff", b"A\xffC", b"acgt", b"a", b"%", b"$", b"A$", b"$A", b"N", b"NN", b"\x00A"]
    qs += [t[p:p + 3] + b"\xff" for p in rng.sample(range(n), min(n, 20))]
    # a suffix of the text plus extra bytes: runs past the end of the text
    for p in sorted({max(0, n - d) for d in (1, 2, 3, 5, 8, 13, 40)}):
        qs += [t[p:] + b"A", t[p:] + b"$", t[p:] + b"\x01", t[p:] + t[p:]]
    # the whole text, with and without an extra byte; the empty query
    qs += [t, t + b"A", b""]
    return qs


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


class Case:
    """One text built every way its spec lists, its reference index and queries, and the expected answers."""

    def __init__(self, S, name, tmp):
        import torch
        text, flags, sources = SPECS[name]
        self.name, self.flags = name, flags
        self.indexes, self._results = [], []
        arrays = None
        try:
            for kind, bits in sources:
                if kind == "built":
                    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
                    args = S.SufrBuilderArgs(text=b"", **flags)
                    r = S.build(args, index_bits=bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
                    r._keep = t
                    self._results.append(r)
                    udt = np.uint32 if bits == 32 else np.uint64  # (the tensors hold the same bits as signed)
                    got = (r.text_tensor().cpu().numpy().tobytes(), r.sa_tensor().cpu().numpy().view(udt),
                           r.lcp_tensor().cpu().numpy().view(udt))
                    index = S.SufrIndex(r, args)
                else:
                    path = tmp / f"{name}_u{bits}.sufr"
                    b = S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(path), **flags), bits)
                    b._res.free()
                    f = parse_sufr(path.read_bytes())
                    assert f.index_bits == bits
                    got = (f.text, f.sa, f.lcp)
                    index = S.SufrIndex.open(path)
                self.indexes.append((f"{kind}_u{bits}", index))
                got = (got[0], got[1].astype(np.int64), got[2].astype(np.int64))
                if arrays is None:
                    arrays = got
                else:  # every source holds the same index
                    assert got[0] == arrays[0] and np.array_equal(got[1], arrays[1]) and np.array_equal(got[2], arrays[2])
        except BaseException:
            self.close()
            raise
        self.ref = R.Index(arrays[0], arrays[1], arrays[2], flags.get("max_query_len") or 0, flags.get("seed_mask"))
        self.caps = run_caps(flags, self.ref.n)
        alphabet = sorted(set(arrays[0])) or [65]
        self.queries = make_queries(self.ref, name, self.caps, alphabet)
        self.full = {m: R.full_ranges(self.ref, self.queries, m) for m in self.caps}

    def expected(self, m, low_memory):
        return R.expected(self.ref, self.queries, m, low_memory, self.full[m])

    def close(self):
        for _, index in self.indexes:
            index.close()
        for r in self._results:
            r.free()
        self.indexes, self._results = [], []


@pytest.fixture(scope="module", params=list(SPECS))
def case(request, S, tmp_path_factory):
    c = Case(S, request.param, tmp_path_factory.mktemp("search_ref"))
    yield c
    c.close()


def _mismatches(queries, got, want, limit=5):
    bad = [(q[:24], g, w) for q, g, w in zip(queries, got, want) if g != w]
    return f"{len(bad)} of {len(queries)} differ, e.g. {bad[:limit]}"


@pytest.mark.gpu
@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
def test_search_count_locate_match_reference(case, low_memory):
    """Every query, every run-time cap, every source of the index: search, count and locate_ranges (ranges and
    hit offsets) equal the host reference."""
    failures = []
    for label, index in case.indexes:
        for m in case.caps:
            want = case.expected(m, low_memory)
            got = index.search(case.queries, max_query_len=m, low_memory=low_memory)
            if got != want:
                failures.append(f"{label} m={m} search: {_mismatches(case.queries, got, want)}")
                continue
            counts = [0 if w is None else w[1] - w[0] for w in want]
            if index.count(case.queries, max_query_len=m, low_memory=low_memory) != counts:
                failures.append(f"{label} m={m} count")
            b, e, ho = index.locate_ranges(case.queries, max_query_len=m, low_memory=low_memory)
            ranges = [None if x == NONE and y == NONE else (int(x), int(y)) for x, y in zip(b, e)]
            if ranges != want:
                failures.append(f"{label} m={m} locate_ranges: {_mismatches(case.queries, ranges, want)}")
            if ho.tolist() != [0] + np.cumsum(counts, dtype=np.int64).tolist():
                failures.append(f"{label} m={m} hit_offsets")
    assert not failures, f"{case.name}:\n" + "\n".join(failures)


@pytest.mark.gpu
def test_zero_cap_answers_like_none(case):
    """A run-time max_query_len of 0 means no run-time cap, on every kind of index and in both memory modes."""
    for label, index in case.indexes:
        for low_memory in (False, True):
            assert index.search(case.queries, max_query_len=0, low_memory=low_memory) == \
                index.search(case.queries, low_memory=low_memory), (label, low_memory)
            b0, e0, h0 = index.locate_ranges(case.queries, max_query_len=0, low_memory=low_memory)
            b1, e1, h1 = index.locate_ranges(case.queries, low_memory=low_memory)
            assert np.array_equal(b0, b1) and np.array_equal(e0, e1) and np.array_equal(h0, h1), (label, low_memory)


@pytest.mark.gpu
@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
@pytest.mark.parametrize("row", LAST_SAMPLED, ids=[f"{c[0]}-m{c[1]}" for c in LAST_SAMPLED])
def test_last_sampled_goldens(S, row, low_memory):
    name, m, q, full, true = row
    idx = S.SufrIndex.open(EXPECTED / name)
    try:
        assert idx.search([q], max_query_len=m, low_memory=low_memory) == [full]
        assert idx.count([q], max_query_len=m, low_memory=low_memory) == [true]
        hits = idx.locate([q], max_query_len=m, low_memory=low_memory)[0]
        assert [h[0] for h in hits] == list(range(*full))
    finally:
        idx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("low", [[], ["--low-memory"]], ids=["in_memory", "low_memory"])
def test_cli_last_sampled(S, low):
    path = str(EXPECTED / "long_dna_sequence.sufr")
    r = subprocess.run([str(EXE), "count", "-m", "6"] + low + [path, "TTTTTT"], capture_output=True, text=True)
    assert (r.returncode, r.stdout) == (0, "TTTTTT 4\n"), r.stderr
    r = subprocess.run([str(EXE), "locate", "-m", "3"] + low + [path, "TTT"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == "TTT" and lines[-1] == "//"
    assert sum(len(ln.rsplit(" ", 1)[1].split(",")) for ln in lines[1:-1]) == 319
    r = subprocess.run([str(EXE), "locate", "-a", "-m", "3"] + low + [path, "TTT"], capture_output=True, text=True)
    assert len(r.stdout.split()) == 1 + 319
