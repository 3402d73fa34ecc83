"""The read side of `.sufr` files: header validation (sufr_b200_file_info), a device index opened from a file
(sufr_b200_index_open), batched locate on the device (sufr_b200_index_locate / _hits) and the `sufr-b200 count` /
`sufr-b200 locate` commands, checked against the reference's own query fixtures run on the reference-written files."""
import ctypes as C
import os
import random
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES, ROOT
from sufrfile import parse_sufr

EXE = ROOT / "sufr_b200" / "sufr-b200"
EXPECTED = GOLDEN / "expected"
QDIR = GOLDEN / "expected_queries"


@pytest.fixture(scope="module")
def S():
    subprocess.check_call(["make", "-C", str(ROOT / "sufr_b200" / "csrc"), "-s", "-j8"])
    import sufr_b200
    return sufr_b200


# ------------------------------------------------------------------ CPU: header validation
@pytest.mark.parametrize("golden", [c[0] for c in GOLDEN_CASES])
def test_file_info_matches_parser(S, golden):
    path = EXPECTED / golden
    want = parse_sufr(path.read_bytes())
    got = S.file_info(path)
    assert got["version"] == want.version == 6
    assert got["index_bits"] == want.index_bits
    for k in ("is_dna", "allow_ambiguity", "ignore_softmask", "text_len", "num_suffixes", "max_query_len",
              "num_sequences", "text_pos", "sa_pos", "lcp_pos", "sequence_starts", "sequence_names", "seed_mask"):
        assert got[k] == getattr(want, k), k
    assert got["file_bytes"] == path.stat().st_size


def _u64(data, off, v):
    data[off:off + 8] = struct.pack("<Q", v)


def _mutations():
    """(id, golden, mutate(bytearray) -> bytes, expected code name, message fragment)"""
    def trunc(n):
        return lambda d: bytes(d[:n])

    def set_u64(off, delta):
        def f(d):
            (v,) = struct.unpack_from("<Q", d, off)
            _u64(d, off, v + delta)
            return bytes(d)
        return f

    def names_count(d):
        f = parse_sufr(bytes(d))
        _u64(d, f.lcp_pos + f.num_suffixes * f.index_bits // 8, f.num_sequences + 1)
        return bytes(d)

    def mask_byte(d):
        f = parse_sufr(bytes(d))
        d[f.text_pos - 2] = 2  # a byte of the mask section
        return bytes(d)

    def unsorted_starts(d):
        # 2.sufr: two u32 starts at offset 60
        a, b = struct.unpack_from("<2I", d, 60)
        struct.pack_into("<2I", d, 60, b, a)
        return bytes(d)

    def version5(d):
        d[0] = 5
        return bytes(d)

    def trailing(d):
        return bytes(d) + b"\0"

    return [
        ("empty", "2.sufr", trunc(0), "ERR_IO", "empty file"),
        ("trunc_1", "2.sufr", trunc(1), "ERR_IO", "truncated header"),
        ("trunc_40", "2.sufr", trunc(40), "ERR_IO", "truncated header"),
        ("trunc_starts", "uniprot.sufr", trunc(200), "ERR_IO", "invalid .sufr file"),
        ("trunc_text", "2.sufr", trunc(90), "ERR_IO", "invalid .sufr file"),
        ("trunc_lcp", "2.sufr", lambda d: bytes(d[:parse_sufr(bytes(d)).lcp_pos + 5]), "ERR_IO", "invalid .sufr file"),
        ("trunc_names", "2.sufr", lambda d: bytes(d[:-2]), "ERR_IO", "sequence names"),
        ("trailing_byte", "2.sufr", trailing, "ERR_IO", "unexpected bytes"),
        ("version5", "2.sufr", version5, "ERR_UNSUPPORTED", "version 5"),
        ("text_pos_plus1", "2.sufr", set_u64(12, 1), "ERR_IO", "text_pos"),
        ("text_pos_minus1", "2.sufr", set_u64(12, -1), "ERR_IO", "text_pos"),
        ("names_count", "2.sufr", names_count, "ERR_IO", "names tail holds 3 names for 2 sequences"),
        ("mask_byte_2", "uniprot-masked.sufr", mask_byte, "ERR_IO", "seed mask byte 2"),
        ("unsorted_starts", "2.sufr", unsorted_starts, "ERR_IO", "strictly increasing"),
        ("suffixes_gt_text", "2.sufr", set_u64(36, 1000), "ERR_IO", "invalid .sufr file"),
        ("width", "2.sufr", set_u64(28, 2), "ERR_IO", "invalid .sufr file"),
    ]


MUTATIONS = _mutations()


@pytest.mark.parametrize("case", MUTATIONS, ids=[m[0] for m in MUTATIONS])
def test_malformed_file_is_refused(S, tmp_path, case):
    from sufr_b200 import _lib
    _, golden, mutate, code, fragment = case
    bad = tmp_path / "bad.sufr"
    bad.write_bytes(mutate(bytearray((EXPECTED / golden).read_bytes())))
    with pytest.raises(S.SufrError) as e:
        S.file_info(bad)
    assert e.value.code == getattr(_lib, code)
    assert str(e.value).startswith(f"{bad}: ")
    assert fragment in str(e.value)


def test_missing_path(S, tmp_path):
    from sufr_b200 import _lib
    p = tmp_path / "nope.sufr"
    with pytest.raises(S.SufrError) as e:
        S.file_info(p)
    assert e.value.code == _lib.ERR_IO
    assert str(e.value) == f"{p}: No such file or directory"  # the writer's "{path}: {io error}" form


def test_u64_file_of_short_text_is_read_by_width(S, tmp_path):
    """--index-bits 64 writes u64 files of short texts: the width comes from the section sizes, not the text length."""
    import oracle as O
    o = O.oracle_build(b"ACGTNNACGT$", is_dna=True, allow_ambiguity=True, index_bits=64, num_partitions=2)
    out = tmp_path / "u64.sufr"
    out.write_bytes(o.file_bytes)
    info = S.file_info(out)
    assert info["index_bits"] == 64 and info["num_suffixes"] == o.num_suffixes
    assert info["sequence_starts"] == [0] and info["sequence_names"] == ["1"]


def test_file_info_struct_layout(S):
    from sufr_b200 import _lib
    src = r'''
    #include "sufr_b200.h"
    #include <stdio.h>
    #include <stddef.h>
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu\n", sizeof(SufrB200FileInfo), offsetof(SufrB200FileInfo, text_len),
             offsetof(SufrB200FileInfo, file_bytes), offsetof(SufrB200FileInfo, seed_mask),
             offsetof(SufrB200FileInfo, sequence_names), offsetof(SufrB200FileInfo, ignore_softmask));
      return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", str(ROOT / "include"), "-o", os.path.join(d, "t"), os.path.join(d, "t.c")])
        out = subprocess.check_output([os.path.join(d, "t")], text=True).split()
    F = _lib.FileInfo
    assert [int(x) for x in out] == [C.sizeof(F), F.text_len.offset, F.file_bytes.offset, F.seed_mask.offset,
                                     F.sequence_names.offset, F.ignore_softmask.offset]


@pytest.mark.parametrize("cmd", ["count", "locate"])
def test_query_cli_surface(S, tmp_path, cmd):
    r = subprocess.run([str(EXE), cmd, "--help"], capture_output=True, text=True)
    assert r.returncode == 0
    for flag in ["--max-query-len", "--low-memory", "--device", "--query-file", "<SUFR>", "[QUERY]..."]:
        assert flag in r.stdout
    assert ("--abs" in r.stdout) == (cmd == "locate")
    r = subprocess.run([str(EXE), cmd], capture_output=True, text=True)  # no file
    assert r.returncode == 2 and "<SUFR>" in r.stderr
    r = subprocess.run([str(EXE), cmd, str(EXPECTED / "2.sufr")], capture_output=True, text=True)  # no query
    assert r.returncode == 2 and "<QUERY>" in r.stderr
    r = subprocess.run([str(EXE), cmd, "--bogus", str(EXPECTED / "2.sufr"), "AC"], capture_output=True, text=True)
    assert r.returncode == 2
    if cmd == "count":
        r = subprocess.run([str(EXE), cmd, "-a", str(EXPECTED / "2.sufr"), "AC"], capture_output=True, text=True)
        assert r.returncode == 2
    bad = tmp_path / "bad.sufr"
    bad.write_bytes(b"\x05" + (EXPECTED / "2.sufr").read_bytes()[1:])
    r = subprocess.run([str(EXE), cmd, str(bad), "AC"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("Error: ") and "version 5" in r.stderr
    r = subprocess.run([str(EXE), cmd, str(tmp_path / "missing.sufr"), "AC"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("Error: ")


def test_top_level_help_lists_the_commands(S):
    for argv, code in (([], 2), (["--help"], 0)):
        r = subprocess.run([str(EXE)] + argv, capture_output=True, text=True)
        assert r.returncode == code
        for cmd in ("create", "count", "locate"):
            assert f"  {cmd}  " in r.stdout
    r = subprocess.run([str(EXE), "create", "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "Commands:" not in r.stdout and "--seed-mask" in r.stdout


def test_unknown_subcommand_lists_the_three(S):
    r = subprocess.run([str(EXE), "extract", "x.sufr"], capture_output=True, text=True)
    assert r.returncode == 2
    assert "'create', 'count' and 'locate'" in r.stderr


# ------------------------------------------------------------------ GPU
def format_locate(queries, hits, absolute):
    """What `sufr-b200 locate` prints, restated from SufrIndex.locate results."""
    lines = []
    for q, hs in zip(queries, hits):
        if absolute:
            lines.append(" ".join([q] + [str(h[1]) for h in hs]))
            continue
        lines.append(q)
        by = {}
        for _, _, name, pos in hs:
            by.setdefault(name.encode(), []).append(pos)
        for name in sorted(by):
            lines.append(name.decode() + " " + ",".join(str(p) for p in sorted(by[name])))
        lines.append("//")
    return "\n".join(lines) + "\n"


# (fixture, file, flags, queries)
CLI_FIXTURES = [
    ("locate1.out", "2.sufr", [], ["AC", "GT"]),
    ("locate-abs.out", "2.sufr", ["-a"], ["AC", "GT"]),
    ("uniprot-search1.out", "uniprot.sufr", [], ["RNELNNEEA", "DTPTNCPT", "GSGLSLLSD"]),
    ("uniprot-search-masked.out", "uniprot-masked.sufr", [], ["RNEL", "DTPT", "GSGL"]),
    ("uniprot-search-masked-mql-3.out", "uniprot-masked.sufr", ["-m", "3"], ["RNELNNEEA", "DTPTNCPT", "GSGLSLLSD"]),
    ("uniprot-search-masked-absolute.out", "uniprot-masked.sufr", ["-a"], ["RNEL"]),
    ("locate_long_dna.out", "long_dna_sequence.sufr", [], ["CATGTTGTCACG", "CCATGGGAC", "GGATGAAGAAAAGCA"]),
    ("locate_long_dna_mql_6.out", "long_dna_sequence.sufr", ["-m", "6"],
     ["CATGTTGTCACG", "CCATGGGAC", "GGATGAAGAAAAGCA"]),
    # locate2.out holds the lines of locate-abs.out followed by one empty line.  No command of the repository is known to
    # print that empty line, so this fixture is compared with its final newline removed; the other eight byte for byte
    ("locate2.out", "2.sufr", ["-a"], ["AC", "GT"]),
]


def _want(fixture):
    text = (QDIR / fixture).read_text()
    return text[:-1] if fixture == "locate2.out" else text


@pytest.mark.gpu
@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
@pytest.mark.parametrize("case", CLI_FIXTURES, ids=[c[0] for c in CLI_FIXTURES])
def test_cli_locate_reproduces_reference_fixtures(S, case, low_memory):
    fixture, sufr, flags, queries = case
    cmd = [str(EXE), "locate"] + flags + (["--low-memory"] if low_memory else []) + [str(EXPECTED / sufr)] + queries
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout == _want(fixture)


@pytest.mark.gpu
@pytest.mark.parametrize("low_memory", [False, True], ids=["in_memory", "low_memory"])
@pytest.mark.parametrize("case", CLI_FIXTURES, ids=[c[0] for c in CLI_FIXTURES])
def test_opened_index_reproduces_reference_fixtures(S, case, low_memory):
    fixture, sufr, flags, queries = case
    mql = int(flags[1]) if flags[:1] == ["-m"] else None
    idx = S.SufrIndex.open(EXPECTED / sufr)
    try:
        hits = idx.locate(queries, max_query_len=mql, low_memory=low_memory)
        assert format_locate(queries, hits, "-a" in flags) == _want(fixture)
    finally:
        idx.close()


@pytest.mark.gpu
def test_cli_query_file_and_counts(S, tmp_path):
    # cli.rs:339-361: `sufr count` -> 2 0 2 on 1.sufr and 1 1 1 on 3.sufr
    for low in ([], ["--low-memory"]):
        r = subprocess.run([str(EXE), "count"] + low + [str(EXPECTED / "1.sufr"), "AC", "X", "GT"], capture_output=True,
                           text=True)
        assert (r.returncode, r.stdout) == (0, "AC 2\nX 0\nGT 2\n"), r.stderr
        qf = tmp_path / "q.txt"
        qf.write_text("AAAAAAA\r\n\nTGTCTC\nTGATAGCAGCTTCTGAACTGGTTACCTGCCGTGAGT")
        r = subprocess.run([str(EXE), "count"] + low + ["-f", str(qf), str(EXPECTED / "3.sufr")], capture_output=True,
                           text=True)
        assert (r.returncode, r.stdout) == (0, "AAAAAAA 1\nTGTCTC 1\nTGATAGCAGCTTCTGAACTGGTTACCTGCCGTGAGT 1\n")
    for low_memory in (False, True):
        idx = S.SufrIndex.open(EXPECTED / "1.sufr")
        assert idx.count(["AC", "X", "GT"], low_memory=low_memory) == [2, 0, 2]
        idx.close()
    # a query without a match: its line and `//` (relative), the query alone (absolute)
    r = subprocess.run([str(EXE), "locate", str(EXPECTED / "2.sufr"), "XX", "AC", "YY"], capture_output=True, text=True)
    assert r.stdout == "XX\n//\nAC\nABC 0,4\nDEF 0,4\n//\nYY\n//\n"
    r = subprocess.run([str(EXE), "locate", "-a", str(EXPECTED / "2.sufr"), "XX", "GT", "YY"], capture_output=True,
                       text=True)
    assert r.stdout == "XX\nGT 15 6 11 2\nYY\n"


def _device_index(S, fasta, flags, index_bits=32):
    import torch
    flags = dict(flags)
    delim = flags.pop("delimiter", b"%")
    seq = S.read_sequence_file(GOLDEN / "inputs" / fasta, delim)
    t = torch.frombuffer(bytearray(seq.seq), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", sequence_starts=seq.start_positions, sequence_names=seq.sequence_names, **flags)
    r = S.build(args, index_bits=index_bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    r._keep = t
    return S.SufrIndex(r, args), r


@pytest.mark.gpu
@pytest.mark.parametrize("golden,fasta,flags", GOLDEN_CASES, ids=[c[0] for c in GOLDEN_CASES])
def test_opened_file_answers_like_a_fresh_build(S, golden, fasta, flags):
    f = parse_sufr((EXPECTED / golden).read_bytes())
    rng = random.Random(golden)
    text = f.text.decode("latin-1")
    queries = []
    for _ in range(300):
        p, ln = rng.randrange(len(text)), rng.randrange(1, 12)
        queries.append(text[p:p + ln])
    alphabet = sorted(set(text))
    queries += ["".join(rng.choice(alphabet) for _ in range(rng.randrange(6, 14))) for _ in range(60)]
    queries += ["#absent", "ZZZZ"]
    opened = S.SufrIndex.open(EXPECTED / golden)
    fresh, r = _device_index(S, fasta, flags)
    try:
        assert opened.info["num_suffixes"] == r.num_suffixes
        for mql in (None, 3):
            for low_memory in (False, True):
                a = opened.search(queries, max_query_len=mql, low_memory=low_memory)
                b = fresh.search(queries, max_query_len=mql, low_memory=low_memory)
                assert a == b, (mql, low_memory)
                assert opened.locate(queries, max_query_len=mql, low_memory=low_memory) == \
                    fresh.locate(queries, max_query_len=mql, low_memory=low_memory), (mql, low_memory)
    finally:
        opened.close()
        fresh.close()
        r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["opened", "built"])
def test_interleaved_search_and_locate_keep_the_right_subsample(S, kind):
    """search() / count() and locate() on ONE index, with run-time max_query_lens that need different LCP-subsampled
    arrays, interleaved: every answer equals that of a fresh index (locate makes its subsample inside the library)."""
    queries = ["CATGTTGTCACG", "CCATGGGAC", "GGATGAAGAAAAGCA", "ACG", "TTT", "GA", "CCCCCC"]

    def fresh():
        if kind == "opened":
            return S.SufrIndex.open(EXPECTED / "long_dna_sequence.sufr"), None
        return _device_index(S, "long_dna_sequence.fa", dict(is_dna=True))

    idx, r = fresh()
    try:
        for op, mql in (("count", 3), ("locate", 6), ("count", 3), ("locate", 3), ("search", 6), ("locate", 6),
                        ("count", 6), ("locate", 3), ("search", 3)):
            want_idx, want_r = fresh()
            try:
                if op == "locate":
                    got, want = idx.locate(queries, max_query_len=mql), want_idx.locate(queries, max_query_len=mql)
                else:
                    got = getattr(idx, op)(queries, max_query_len=mql)
                    want = getattr(want_idx, op)(queries, max_query_len=mql)
                assert got == want, (op, mql)
            finally:
                want_idx.close()
                if want_r is not None:
                    want_r.free()
    finally:
        idx.close()
        if r is not None:
            r.free()


@pytest.mark.gpu
def test_u64_file_answers_like_u32(S, tmp_path):
    seq = S.read_sequence_file(GOLDEN / "inputs" / "long_dna_sequence.fa", b"%")
    files = {}
    for bits in (32, 64):
        path = tmp_path / f"u{bits}.sufr"
        args = S.SufrBuilderArgs(text=seq.seq, path=str(path), is_dna=True, sequence_starts=seq.start_positions,
                                 sequence_names=seq.sequence_names)
        S.SufrBuilder(args, bits)
        files[bits] = path
    assert S.file_info(files[64])["index_bits"] == 64
    queries = ["CATGTTGTCACG", "CCATGGGAC", "GGATGAAGAAAAGCA", "ACG", "T", "NNNN"]
    a, b = S.SufrIndex.open(files[32]), S.SufrIndex.open(files[64])
    try:
        for mql in (None, 6):
            for low in (False, True):
                assert a.locate(queries, mql, low) == b.locate(queries, mql, low)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_device_locate_against_numpy(S, tmp_path):
    """200 kbp of ~1000 records: 20 k queries (1-4-mers with thousands of hits each included) through locate + hit
    windows that split queries, against an SA gather + searchsorted over the sequence starts."""
    from sufr_b200 import _lib
    rng = np.random.default_rng(3)
    lens = rng.integers(50, 350, 1000)
    recs = [bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(n))]) for n in lens]
    text = b"%".join(recs) + b"$"
    starts = np.concatenate([[0], np.cumsum(lens[:-1] + 1)]).astype(np.uint64)
    names = [f"r{i:04d}" for i in range(len(recs))]
    path = tmp_path / "many.sufr"
    S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(path), is_dna=True, sequence_starts=starts.tolist(),
                                    sequence_names=names), 32)
    sa = parse_sufr(path.read_bytes()).sa.astype(np.uint64)
    pyr = random.Random(4)
    tx = text.decode()
    queries = ["".join(pyr.choice("ACGT") for _ in range(pyr.randrange(1, 5))) for _ in range(200)]
    for _ in range(14_800):
        p = pyr.randrange(len(tx) - 30)
        queries.append(tx[p:p + pyr.randrange(5, 25)])
    queries += ["".join(pyr.choice("ACGT") for _ in range(pyr.randrange(12, 20))) for _ in range(5_000)]
    idx = S.SufrIndex.open(path)
    try:
        b, e, ho = idx.locate_ranges(queries, low_memory=True)
        none = np.uint64(0xFFFFFFFFFFFFFFFF)
        counts = np.where(b == none, 0, e - b).astype(np.uint64)
        assert np.array_equal(ho, np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64))
        assert counts[:200].min() > 100  # the short queries have many hits
        for i in list(range(0, 200, 7)) + list(range(200, len(queries), 311)):  # counts vs a scan of the text
            q, n, k = queries[i], 0, tx.find(queries[i])
            while k >= 0:
                n, k = n + 1, tx.find(q, k + 1)
            assert counts[i] == n, (q, counts[i], n)
        # restatement of every hit
        qidx = np.repeat(np.arange(len(queries)), counts.astype(np.int64))
        rank = b[qidx] + (np.arange(int(ho[-1]), dtype=np.uint64) - ho[qidx])
        suf = sa[rank.astype(np.int64)]
        seqi = np.searchsorted(starts, suf, side="right") - 1
        total = int(ho[-1])
        cuts = sorted({0, 7, int(ho[3]) + 1, total // 3, total // 2 + 5, total - 1, total})
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            s_, q_, p_ = idx.hits(lo, hi - lo)
            assert np.array_equal(s_, suf[lo:hi])
            assert np.array_equal(q_, seqi[lo:hi].astype(np.uint64))
            assert np.array_equal(p_, suf[lo:hi] - starts[seqi[lo:hi]])
        assert [len(x) for x in idx.hits(total, 0)] == [0, 0, 0]
        for first, count in ((total, 1), (total - 1, 2), (total + 1, 0)):
            with pytest.raises(S.SufrError) as ex:
                idx.hits(first, count)
            assert ex.value.code == _lib.ERR_ARGUMENT
        # the list form keeps SufrFile::locate's contract
        got = idx.locate(queries[:50])
        for i, hs in enumerate(got):
            assert [h[0] for h in hs] == list(range(int(b[i]), int(e[i])))
            assert all(tx[h[1]:h[1] + len(queries[i])] == queries[i] for h in hs)
            assert all(starts[names.index(h[2])] + h[3] == h[1] for h in hs)
    finally:
        idx.close()


@pytest.mark.gpu
def test_index_without_sequence_starts(S):
    import torch
    text = b"ACGTACGTACGT$"
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", is_dna=True, sequence_starts=(), sequence_names=())
    r = S.build(args, index_bits=32, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    idx = S.SufrIndex(r, args)
    try:
        (hs,) = idx.locate(["CGT"])
        assert sorted(h[1] for h in hs) == [1, 5, 9]
        assert all(h[2] is None and h[3] == h[1] for h in hs)
    finally:
        idx.close()
        r.free()


@pytest.mark.gpu
def test_suffix_array_entry_beyond_text_is_refused(S, tmp_path):
    from sufr_b200 import _lib
    data = bytearray((EXPECTED / "2.sufr").read_bytes())
    f = parse_sufr(bytes(data))
    struct.pack_into("<I", data, f.sa_pos + 4 * 3, f.text_len)
    bad = tmp_path / "bad_sa.sufr"
    bad.write_bytes(bytes(data))
    assert S.file_info(bad)["num_suffixes"] == f.num_suffixes  # the header is intact
    with pytest.raises(S.SufrError) as e:
        S.SufrIndex.open(bad)
    assert e.value.code == _lib.ERR_IO and "suffix array entry" in str(e.value)
    r = subprocess.run([str(EXE), "count", str(bad), "AC"], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("Error: ")
