"""SURVEY 8(f) rank 4: the read side that consumes the LCP array -- LCP-subsampled suffix array and batched search on
the GPU -- against the reference's own query fixtures (data/expected/*.out, copied to tests/golden/expected_queries;
commands from sufr/tests/cli.rs:305-350 and :873-1123) and against a brute-force scan of the text."""
import random

import numpy as np
import pytest

from conftest import GOLDEN
from index_matrix import device_index
import oracle as O

pytestmark = pytest.mark.gpu
QDIR = GOLDEN / "expected_queries"


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


def make_index(S, fasta, index_bits=32, delimiter=b"%", **kw):
    seq = S.read_sequence_file(GOLDEN / "inputs" / fasta, delimiter)
    return device_index(S, seq.seq, seq.start_positions, seq.sequence_names, index_bits, **kw) + (seq,)


def parse_relative(path):
    """`sufr locate` output: query / 'name pos,pos' lines / '//' (sufr/src/lib.rs:506-530)."""
    out, cur, q = {}, None, None
    for line in path.read_text().splitlines():
        if line == "//":
            q = None
        elif q is None:
            q = line
            out[q] = {}
        else:
            name, positions = line.rsplit(" ", 1)
            out[q][name] = [int(x) for x in positions.split(",")]
    return out


def relative(hits):
    d = {}
    for _, _, name, pos in sorted(hits, key=lambda h: (h[2], h[3])):
        d.setdefault(name, []).append(pos)
    return d


@pytest.mark.parametrize("low_memory", [False, True])
def test_count_fixtures(S, low_memory):
    # cli.rs:339-361: `sufr count 1.sufr AC X GT` -> 2 0 2; 3.sufr -> 1 1 1
    idx, r, _ = make_index(S, "1.fa", is_dna=True)
    assert idx.count(["AC", "X", "GT"], low_memory=low_memory) == [2, 0, 2]
    idx.close(); r.free()
    idx, r, _ = make_index(S, "3.fa", is_dna=True)
    assert idx.count(["AAAAAAA", "TGTCTC", "TGATAGCAGCTTCTGAACTGGTTACCTGCCGTGAGT"], low_memory=low_memory) == [1, 1, 1]
    idx.close(); r.free()


LOCATE_CASES = [
    # (input, build flags, queries, run-time max_query_len, fixture)           cli.rs
    ("2.fa", dict(is_dna=True), ["AC", "GT"], None, "locate1.out"),                                     # :907-928
    ("uniprot.fa", dict(), ["RNELNNEEA", "DTPTNCPT", "GSGLSLLSD"], None, "uniprot-search1.out"),        # :949-975
    ("uniprot.fa", dict(seed_mask="10111011"), ["RNEL", "DTPT", "GSGL"], None, "uniprot-search-masked.out"),  # :978-1026
    ("uniprot.fa", dict(seed_mask="10111011"), ["RNELNNEEA", "DTPTNCPT", "GSGLSLLSD"], 3,
     "uniprot-search-masked-mql-3.out"),                                                                  # :1029-1046
    ("long_dna_sequence.fa", dict(is_dna=True), ["CATGTTGTCACG", "CCATGGGAC", "GGATGAAGAAAAGCA"], None,
     "locate_long_dna.out"),                                                                              # :1066-1093
    ("long_dna_sequence.fa", dict(is_dna=True), ["CATGTTGTCACG", "CCATGGGAC", "GGATGAAGAAAAGCA"], 6,
     "locate_long_dna_mql_6.out"),                                                                        # :1096-1123
]


@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
@pytest.mark.parametrize("case", LOCATE_CASES, ids=[c[4] for c in LOCATE_CASES])
def test_locate_fixtures(S, case, low_memory):
    """The reference runs every locate test in its three memory modes and expects the same output (cli.rs:873-903):
    in-memory (LCP-subsampled array when -m is shorter than the build's) and low-memory (full array)."""
    fasta, kw, queries, mql, fixture = case
    idx, r, _ = make_index(S, fasta, **kw)
    try:
        want = parse_relative(QDIR / fixture)
        got = idx.locate(queries, max_query_len=mql, low_memory=low_memory)
        assert {q: relative(h) for q, h in zip(queries, got)} == want
    finally:
        idx.close(); r.free()


@pytest.mark.parametrize("fasta,kw,queries,fixture", [
    ("2.fa", dict(is_dna=True), ["AC", "GT"], "locate-abs.out"),                                    # cli.rs:931-946
    ("uniprot.fa", dict(seed_mask="10111011"), ["RNEL"], "uniprot-search-masked-absolute.out"),     # cli.rs:1049-1063
])
def test_locate_absolute_fixtures(S, fasta, kw, queries, fixture):
    """`locate -a` prints the suffixes in RANK order: pins the rank range and the suffix array together."""
    idx, r, _ = make_index(S, fasta, **kw)
    try:
        got = idx.locate(queries)
        lines = [q + " " + " ".join(str(h[1]) for h in hits) for q, hits in zip(queries, got)]
        assert "\n".join(lines) + "\n" == (QDIR / fixture).read_text()
    finally:
        idx.close(); r.free()


def test_subsample_matches_definition(S):
    """sufr_file.rs:443-453 / lib.rs:167-216: entries with lcp < max_query_len, and their ranks."""
    idx, r, _ = make_index(S, "long_dna_sequence.fa", is_dna=True)
    try:
        sa = r.sa_tensor().cpu().numpy().astype(np.uint32)
        lcp = r.lcp_tensor().cpu().numpy().astype(np.uint32)
        for q in (1, 3, 6, 12, 10_000):
            kept = idx.subsample(q)
            assert kept == int((lcp < q).sum())
    finally:
        idx.close(); r.free()


@pytest.mark.parametrize("bits", [32, 64])
def test_batched_search_against_brute_force(S, bits):
    """20 000 queries in one launch (present substrings and random strings), with and without a run-time cap."""
    import torch
    rng = random.Random(bits)
    text = "".join(rng.choice("ACGT") for _ in range(200_000)) + "$"
    t = torch.frombuffer(bytearray(text.encode()), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", is_dna=True)
    r = S.build(args, index_bits=bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    idx = S.SufrIndex(r, args)
    try:
        queries = []
        for _ in range(10_000):
            p, ln = rng.randrange(len(text) - 40), rng.randrange(1, 24)
            queries.append(text[p:p + ln])
        queries += ["".join(rng.choice("ACGT") for _ in range(rng.randrange(8, 16))) for _ in range(10_000)]
        counts = idx.count(queries, low_memory=True)
        for q, c in list(zip(queries, counts))[::97]:
            n, k = 0, text.find(q)
            while k >= 0:
                n, k = n + 1, text.find(q, k + 1)
            assert c == n, (q, c, n)
        # a run-time max_query_len of 8: hits = occurrences of the first 8 characters
        capped = idx.search(queries[:2000], max_query_len=8, low_memory=True)
        for q, rr in list(zip(queries[:2000], capped))[::53]:
            n, k = 0, text.find(q[:8])
            while k >= 0:
                n, k = n + 1, text.find(q[:8], k + 1)
            assert (0 if rr is None else rr[1] - rr[0]) == n, (q, rr, n)
        # The in-memory mode searches the LCP-subsampled array and maps back through the sampled ranks exactly as
        # sufr_search.rs:119-136 does: the range ends at the LAST SAMPLED entry + 1 when more than one sampled entry
        # matches (so the tail run of that entry is not counted), and at the next sampled rank when only one does.
        lcp = r.lcp_tensor().cpu().numpy().astype(np.int64)
        sampled = np.flatnonzero(lcp < 8)
        sub = idx.search(queries[:2000], max_query_len=8, low_memory=False)
        for full, got in zip(capped, sub):
            if full is None:
                assert got is None
                continue
            lo, hi = np.searchsorted(sampled, full[0]), np.searchsorted(sampled, full[1]) - 1
            assert sampled[lo] == full[0]
            if lo == hi:
                want_end = len(lcp) if lo == len(sampled) - 1 else int(sampled[lo + 1])
                assert want_end == full[1]
            else:
                want_end = int(sampled[hi]) + 1
            assert got == (full[0], want_end), (full, got)
    finally:
        idx.close(); r.free()
