"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference's golden files.
Bit-exact: SA, LCP, transformed text, and the whole `.sufr` file."""
import random
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES
import oracle as O
from sufrfile import parse_sufr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


def seed_of(*parts) -> int:
    """Deterministic seed (Python's hash() of str is randomised per process)."""
    return zlib.crc32(repr(parts).encode())


def gpu_vs_oracle(S, text, index_bits=32, **kw):
    # few partitions on tiny texts: the reference (and so the oracle) cannot draw more distinct ACGT$ pivots
    # than the text has (it would loop forever, sufr_builder.rs:787-796)
    parts = kw.pop("oracle_partitions", 16 if len(text) > 2000 else 1)
    want = O.oracle_build(text, num_partitions=parts, threads=4, index_bits=index_bits, **kw)
    got = S.build(S.SufrBuilderArgs(text=text, **kw), index_bits=index_bits)
    try:
        assert got.text == want.text
        assert got.num_suffixes == want.num_suffixes
        sa, lcp = got.sa.copy(), got.lcp.copy()
        assert sa.dtype == want.sa.dtype
        if not np.array_equal(sa, want.sa):
            bad = int(np.nonzero(sa != want.sa)[0][0])
            raise AssertionError(f"SA differs first at rank {bad}: got {sa[bad:bad+5]} want {want.sa[bad:bad+5]}")
        if not np.array_equal(lcp, want.lcp):
            bad = int(np.nonzero(lcp != want.lcp)[0][0])
            raise AssertionError(f"LCP differs first at rank {bad}: got {lcp[bad:bad+5]} want {want.lcp[bad:bad+5]} "
                                 f"(sa {sa[max(0,bad-1):bad+1]})")
        assert got.n_ranges == want.n_ranges
        return got.timings, got.c.refine_rounds, got.c.doubling_rounds
    finally:
        got.free()


@pytest.mark.parametrize("golden,fasta,flags", GOLDEN_CASES, ids=[c[0] for c in GOLDEN_CASES])
def test_golden_whole_file(S, tmp_path, golden, fasta, flags):
    """The reference's own create tests (sufr/tests/cli.rs:113-302) compare the SA; we compare the file."""
    flags = dict(flags)
    delim = flags.pop("delimiter", b"%")
    seq = S.read_sequence_file(GOLDEN / "inputs" / fasta, delim)
    out = tmp_path / golden
    b = S.SufrBuilder(S.SufrBuilderArgs(text=seq.seq, path=str(out), sequence_starts=seq.start_positions,
                                        sequence_names=seq.sequence_names, **flags), 32)
    want = (GOLDEN / "expected" / golden).read_bytes()
    g = parse_sufr(want)
    assert b.text == g.text
    np.testing.assert_array_equal(b.suffix_array, g.sa)
    np.testing.assert_array_equal(b.lcp_array, g.lcp)
    assert out.read_bytes() == want
    assert b.num_suffixes == g.num_suffixes


def test_lib_rs_vectors(S):
    # libsufr/src/lib.rs:45-92 (u32) and :94-140 (u64)
    d = S.read_sequence_file(GOLDEN / "inputs" / "2.fa", b"N")
    r = S.build(S.SufrBuilderArgs(text=d.seq, is_dna=True, num_partitions=2, random_seed=0), index_bits=32)
    assert r.text == b"ACGTACGTNACGTACGT$"
    assert r.sa.tolist() == [17, 13, 9, 0, 4, 14, 10, 1, 5, 15, 11, 2, 6, 16, 12, 3, 7]
    assert r.lcp.tolist() == [0, 0, 4, 8, 4, 0, 3, 7, 3, 0, 2, 6, 2, 0, 1, 5, 1]
    d = S.read_sequence_file(GOLDEN / "inputs" / "1.fa", b"N")
    r = S.build(S.SufrBuilderArgs(text=d.seq, is_dna=True, allow_ambiguity=True, num_partitions=2, random_seed=0),
                index_bits=64)
    assert r.sa.dtype == np.uint64
    assert r.sa.tolist() == [10, 6, 0, 7, 1, 8, 2, 5, 4, 9, 3]
    assert r.lcp.tolist() == [0, 0, 4, 0, 3, 0, 2, 0, 1, 0, 1]


@pytest.mark.parametrize("fasta,mask,want", [
    ("mostlya1.fa", "101", [7, 6, 5, 4, 2, 0, 1, 3]),
    ("mostlya2.fa", "11011", [16, 13, 9, 5, 1, 12, 8, 4, 0, 14, 10, 6, 2, 15, 11, 7, 3]),
    ("spaced_input.fa", "11000111",
     [42, 18, 12, 0, 32, 29, 13, 23, 21, 6, 40, 1, 33, 19, 30, 10, 28, 9, 17, 14, 4, 26, 39, 22, 25, 38, 24,
      35, 7, 36, 15, 41, 5, 20, 31, 11, 27, 8, 16, 3, 37, 34, 2]),
])
def test_lib_rs_spaced_seeds(S, fasta, mask, want):
    # libsufr/src/lib.rs:221-365: pins the position-descending tie order
    d = S.read_sequence_file(GOLDEN / "inputs" / fasta, b"N")
    r = S.build(S.SufrBuilderArgs(text=d.seq, is_dna=True, num_partitions=1, random_seed=0, seed_mask=mask))
    assert r.sa.tolist() == want


def rand_text(rng, n, alphabet, repeat_p=0.0, max_rep=40):
    out = bytearray()
    while len(out) < n:
        if out and rng.random() < repeat_p:
            s = rng.randrange(len(out))
            ln = rng.randrange(1, max_rep)
            out += out[s:s + ln]
        else:
            out.append(rng.choice(alphabet))
    return bytes(out[:n]) + b"$"


ALPHABETS = {
    "acgt": (b"ACGT", dict(is_dna=True)),
    "dna_mixed": (b"ACGTNacgtn%RY", dict(is_dna=True)),
    "dna_amb": (b"ACGTNacgtn%RY", dict(is_dna=True, allow_ambiguity=True)),
    "dna_soft": (b"ACGTNacgtn%", dict(is_dna=True, ignore_softmask=True)),
    "dna_amb_soft": (b"ACGTNacgtn%", dict(is_dna=True, allow_ambiguity=True, ignore_softmask=True)),
    "protein": (b"ACDEFGHIKLMNPQRSTVWY%", dict()),
    "binary": (b"AB", dict()),
    "bytes": (bytes(range(1, 36)) + bytes(range(128, 250)), dict()),
    # both sides of the lowercase range 97..122, and the same bytes with bit 7 set (4-bytes-at-a-time transform)
    "case_edges": (bytes([0x40, 0x41, 0x5A, 0x5B, 0x60, 0x61, 0x6E, 0x7A, 0x7B, 0x7F, 0x80, 0xC1, 0xE1, 0xFA, 0xFF]), dict()),
    "case_edges_soft": (bytes([0x40, 0x41, 0x5A, 0x5B, 0x60, 0x61, 0x6E, 0x7A, 0x7B, 0x7F, 0x80, 0xC1, 0xE1, 0xFA, 0xFF]),
                        dict(ignore_softmask=True)),
}


@pytest.mark.parametrize("name", list(ALPHABETS))
@pytest.mark.parametrize("n", [1, 2, 5, 63, 64, 65, 1000, 30000])
def test_full_sort_random(S, name, n):
    alphabet, flags = ALPHABETS[name]
    rng = random.Random(seed_of(name, n))
    text = rand_text(rng, n, alphabet, repeat_p=0.05)
    if n <= 2:
        text = text[:-1] + b"$$$"[: 4 - n]  # the reference needs text_len >= 4 (partition count n/4)
    gpu_vs_oracle(S, text, **flags)


@pytest.mark.parametrize("mask", ["101", "1101", "11011", "10111011", "1101101101", "111010010100110111",
                                  "1" * 20 + "0" + "1" * 20])
@pytest.mark.parametrize("name", ["acgt", "dna_amb", "protein", "binary"])
def test_seed_mask_random(S, mask, name):
    alphabet, flags = ALPHABETS[name]
    rng = random.Random(seed_of(mask, name))
    text = rand_text(rng, rng.randrange(50, 20000), alphabet, repeat_p=0.05)
    gpu_vs_oracle(S, text, seed_mask=mask, **flags)


@pytest.mark.parametrize("kw", [dict(), dict(max_query_len=0), dict(seed_mask="1" * 14 + "0" + "1" * 6),
                                dict(is_dna=True, allow_ambiguity=True)], ids=["protein", "mql", "mask", "dna_amb"])
def test_general_path_full_word_first_sort(S, kw, monkeypatch):
    """The general path normally sorts log2(n)+8 key bits first and refines the rest; the whole-word first sort
    it replaces must give the same result."""
    rng = random.Random(seed_of("full_word", str(kw)))
    alphabet = b"ACGTN" if kw.get("is_dna") else b"ACDEFGHIKLMNPQRSTVWY"
    kw = dict(kw)
    if "max_query_len" in kw:  # a cap above every LCP: no ties, so the reference's result is well defined
        text = rand_text(rng, 40000, alphabet)
        kw["max_query_len"] = int(O.oracle_build(text, num_partitions=4).lcp.max()) + 1
    else:
        text = rand_text(rng, 40000, alphabet, repeat_p=0.05)
    gpu_vs_oracle(S, text, **kw)
    monkeypatch.setenv("SUFR_B200_DEBUG_FULL_WORD_SORT", "1")
    gpu_vs_oracle(S, text, **kw)


def test_text_without_sentinel(S):
    # library users may pass a text without a trailing '$' (sufr_builder.rs:1044, 1086)
    for t in (b"TTTAGC", b"ACGTNNACGT", b"AAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA"):
        gpu_vs_oracle(S, t)
        gpu_vs_oracle(S, t, seed_mask="101")


@pytest.mark.parametrize("unit,copies", [(b"A", 3000), (b"AC", 2500), (b"ACGGT", 1500), (b"ACGTTGCATTGACCA", 700)])
def test_tandem_repeats_use_prefix_doubling(S, unit, copies):
    """Long-LCP worst case (BASELINE config 5 flavour): deep repeats switch to prefix doubling."""
    rng = random.Random(len(unit))
    text = rand_text(rng, 500, b"ACGT") [:-1] + unit * copies + rand_text(rng, 300, b"ACGT")[:-1] + unit * (copies // 2) + b"$"
    _, _, doubling = gpu_vs_oracle(S, text, is_dna=True)
    assert doubling > 0
    gpu_vs_oracle(S, text, is_dna=True, index_bits=64)


def test_sorted_inverse_suffix_array(S, monkeypatch):
    """Texts above 2^26 bytes fill the inverse suffix array by sorting (position, rank) on the top position bits and
    placing chunks in shared memory; forced here on small texts (one and two radix passes, a partial last chunk)."""
    monkeypatch.setenv("SUFR_B200_DEBUG_SORT_ISA", "1")
    rng = random.Random(11)
    text = rand_text(rng, 30_000, b"ACGT")[:-1] + b"ACGGT" * 6000 + rand_text(rng, 9000, b"ACGT", repeat_p=0.3, max_rep=400)[:-1] \
        + b"ACGGT" * 2500 + b"$"
    _, _, doubling = gpu_vs_oracle(S, text, is_dna=True)
    assert doubling > 0
    gpu_vs_oracle(S, text, is_dna=True, index_bits=64)
    gpu_vs_oracle(S, text)
    big = rand_text(rng, 200_000, b"ACGT")[:-1] + b"AACCGGTTAC" * 9000 + b"$"   # 18 position bits: two passes
    _, _, doubling = gpu_vs_oracle(S, big, is_dna=True)
    assert doubling > 0


def n_run_text(rng, runs, filler=400):
    parts = []
    for r in runs:
        parts.append(rand_text(rng, rng.randrange(50, filler), b"ACGT")[:-1])
        parts.append(b"N" * r)
    parts.append(rand_text(rng, 200, b"ACGT")[:-1])
    return b"".join(parts) + b"$"


@pytest.mark.parametrize("runs", [[1000], [999], [2000], [1500, 1500, 1200, 3000], [1000, 1000, 1000, 1000, 1000, 1000]])
@pytest.mark.parametrize("soft", [False, True])
def test_long_n_runs_allow_ambiguity(S, runs, soft):
    """SURVEY 8a rule 3: every N-prefixed suffix lies in a recorded (>= 1000) run, or there is a single
    short run, so the reference result is a function of the input."""
    rng = random.Random(sum(runs) + soft)
    text = n_run_text(rng, runs)
    if soft:
        text = text.replace(b"N", b"n")
    gpu_vs_oracle(S, text, is_dna=True, allow_ambiguity=True, ignore_softmask=soft)
    # same text without --allow-ambiguity: N starts are filtered out, LCPs span the removed stretch
    gpu_vs_oracle(S, text, is_dna=True, ignore_softmask=soft)


@pytest.mark.parametrize("seed", range(3))
def test_max_query_len_without_ties(S, seed):
    rng = random.Random(seed)
    text = rand_text(rng, 5000, b"ACDEFGHIKLMNPQRSTVWY")
    full = O.oracle_build(text, num_partitions=4)
    q = int(full.lcp.max()) + 1
    gpu_vs_oracle(S, text, max_query_len=q)
    gpu_vs_oracle(S, text, max_query_len=q + 100)


@pytest.mark.parametrize("q", [1, 2, 3, 7, 12, 13, 40])
def test_max_query_len_with_ties_properties(S, q):
    """With ties the reference output depends on its merge schedule (SURVEY 8a rule 4); what is defined:
    the first Q bytes are non-decreasing, LCP values < Q are exact, the others are >= Q (we emit exactly Q
    and order ties by descending position)."""
    rng = random.Random(q)
    text = rand_text(rng, 20000, b"ACGT", repeat_p=0.1)
    got = S.build(S.SufrBuilderArgs(text=text, max_query_len=q))
    sa, lcp = got.sa.copy(), got.lcp.copy()
    t, spec_sa, spec_lcp = O.spec_build(text, max_query_len=q)
    assert sa.tolist() == spec_sa
    assert lcp.tolist() == spec_lcp
    ref = O.oracle_build(text, max_query_len=q, num_partitions=4)
    small = ref.lcp < q
    keys_ref = [t[p:p + q] for p in ref.sa.tolist()]
    keys_got = [t[p:p + q] for p in sa.tolist()]
    assert keys_ref == keys_got
    assert np.array_equal(lcp[small], ref.lcp[small])
    assert (lcp[~small] == q).all() and (ref.lcp[~small] >= q).all()


def test_argument_errors(S):
    # same message texts as the reference (sufr_builder.rs:163-165, types.rs:81-83)
    with pytest.raises(S.SufrError, match="Cannot use max_query_len and seed_mask together"):
        S.build(S.SufrBuilderArgs(text=b"ACGT$", max_query_len=3, seed_mask="101"))
    with pytest.raises(S.SufrError, match="Invalid seed mask '111'"):
        S.build(S.SufrBuilderArgs(text=b"ACGT$", seed_mask="111"))


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("kw", [dict(is_dna=True), dict(is_dna=True, seed_mask="1101101101"), dict(),
                                dict(is_dna=True, allow_ambiguity=True)], ids=["dna", "mask", "protein", "amb"])
def test_key_range_shards_concatenate(S, world, kw):
    """Multi-GPU decomposition, emulated on one device: shard r of `world` for every r, seams repaired,
    concatenation == the unsharded oracle result."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = random.Random(world)
    alphabet = b"ACDEFGHIKLMNPQRSTVWY%" if not kw else b"ACGTN%"
    text = rand_text(rng, 50000, alphabet, repeat_p=0.03)
    want = O.oracle_build(text, num_partitions=16, threads=4, **kw)
    shards = [S.build(S.SufrBuilderArgs(text=text, **kw), rank=r, world_size=world) for r in range(world)]
    meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
    offs, total = shard_layout(meta)
    assert total == want.num_suffixes
    for r, s in enumerate(shards):
        s.set_shard_layout(offs[r], total)
        prev = previous_last_suffix(meta, r)
        if prev is not None and s.num_suffixes:
            s.patch_seam(prev)
    sa = np.concatenate([s.sa for s in shards])
    lcp = np.concatenate([s.lcp for s in shards])
    assert np.array_equal(sa, want.sa)
    assert np.array_equal(lcp, want.lcp)
    assert sum(1 for s in shards if s.num_suffixes) >= min(world, 2)


@pytest.mark.parametrize("world", [4, 16, 64])
@pytest.mark.parametrize("general_path", [False, True], ids=["fast2", "3bit"])
def test_shards_keep_n_run_tie_chains_together(S, monkeypatch, world, general_path):
    """N-run tie rule (sufr_builder.rs:305-307, :701-712) under sharding: many recorded runs (>= 1000 N) that end in
    the same base make long chains of equal (remaining run length, next byte) -- suffixes N^r A.. with r = 1..3 fall
    into different 12-bit histogram bins, so a key-range cut between the 'NA??' bins would split a chain and the
    concatenated shards would differ from the unsharded (and the reference's) order.  With many shards the cuts land
    everywhere; no cut may fall inside the N-prefixed key range."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    if general_path:
        monkeypatch.setenv("SUFR_B200_DEBUG_NO_FAST2", "1")
    rng = np.random.default_rng(world)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    parts = []
    for k in range(40):
        parts.append(acgt[rng.integers(0, 4, int(rng.integers(20, 200)))])
        parts.append(np.full(1000 + (k % 3), ord("N"), dtype=np.uint8))  # runs of 1000..1002 N
        parts.append(np.frombuffer(b"A", dtype=np.uint8))                 # all followed by the same base
        parts.append(acgt[rng.integers(0, 4, 3)])                          # and then different continuations
    text = np.concatenate(parts).tobytes() + b"$"
    kw = dict(is_dna=True, allow_ambiguity=True)
    want = O.oracle_build(text, num_partitions=16, threads=4, **kw)
    assert len(want.n_ranges) == 40
    shards = [S.build(S.SufrBuilderArgs(text=text, **kw), rank=r, world_size=world) for r in range(world)]
    try:
        meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
        offs, total = shard_layout(meta)
        assert total == want.num_suffixes
        for r, s in enumerate(shards):
            s.set_shard_layout(offs[r], total)
            prev = previous_last_suffix(meta, r)
            if prev is not None and s.num_suffixes:
                s.patch_seam(prev)
        sa = np.concatenate([s.sa for s in shards])
        lcp = np.concatenate([s.lcp for s in shards])
        assert np.array_equal(sa, want.sa)
        assert np.array_equal(lcp, want.lcp)
    finally:
        for s in shards:
            s.free()


def test_sequence_names_must_match_starts(S):
    with pytest.raises(S.SufrError, match="sequence_names has 1 entries but sequence_starts has 2"):
        S.build(S.SufrBuilderArgs(text=b"ACGT%ACGT$", sequence_starts=[0, 5], sequence_names=["a"]))


def test_device_resident_result_and_text(S):
    """The bench's device-resident path: text already in HBM, SA/LCP left in HBM."""
    import torch
    rng = np.random.default_rng(3)
    text = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 300000)].tobytes() + b"$"
    want = O.oracle_build(text, is_dna=True, threads=4)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    for bits, tdt in ((32, torch.int32), (64, torch.int64)):
        r = S.build(S.SufrBuilderArgs(text=b"", is_dna=True), index_bits=bits, result_memory=S.MEM_DEVICE,
                    device_text=(d_text.data_ptr(), d_text.numel()))
        assert r.on_device and r.num_suffixes == want.num_suffixes
        sa = r.sa_tensor().cpu().numpy().astype(np.uint64) & (0xFFFFFFFF if bits == 32 else 0xFFFFFFFFFFFFFFFF)
        lcp = r.lcp_tensor().cpu().numpy().astype(np.uint64) & (0xFFFFFFFF if bits == 32 else 0xFFFFFFFFFFFFFFFF)
        assert bytes(r.text_tensor().cpu().numpy().tobytes()) == want.text
        assert np.array_equal(sa, want.sa.astype(np.uint64))
        assert np.array_equal(lcp, want.lcp.astype(np.uint64))
        r.free()


def test_bench_workload_generator_matches_cpu_restatement(S):
    """bench.py's synthetic text: GPU kernel == numpy restatement (the CPU baseline runs on a prefix)."""
    import torch
    import bench
    from sufr_b200 import _lib
    text_len, starts = bench.record_layout(3_000_000)
    ctx = S.default_context(0)
    d = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    st = np.asarray(starts, dtype=np.uint64)
    assert _lib.lib().sufr_b200_synth_dna(ctx.handle, d.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                          ord("%")) == 0
    got = d.cpu().numpy().tobytes()
    assert got == bench.synth_prefix_numpy(text_len, text_len, starts)
    assert got.count(b"%") == 23 and got.endswith(b"$")


@pytest.mark.parametrize("bits", [32, 64])
def test_bench_dump_outputs_match_oracle(tmp_path, bits):
    """`bench.py --dump-outputs`: the sampled suffix array, LCP array and text of the last timed step are the oracle's
    at the dumped ranks and positions, and --steps sets the number of timed steps."""
    import json
    import subprocess
    import sys
    import bench
    from conftest import ROOT
    bases = 2_000_000  # more suffixes than bench.DUMP_SAMPLE: the sampled path
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--bases", str(bases), "--index-bits", str(bits),
                        "--steps", "2", "--warmup", "3", "--no-configs", "--no-e2e", "--no-cpu",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["verify"]["ok"]
    text_len, starts = bench.record_layout(bases)
    want = O.oracle_build(bench.synth_prefix_numpy(text_len, text_len, starts), is_dna=True, threads=8, index_bits=bits)
    d = {f.stem: np.load(f) for f in tmp_path.glob("*.npy")}
    assert d["sizes"].tolist() == [want.num_suffixes, text_len]
    assert d["sa"].dtype == np.float64 and d["text"].dtype == np.float32
    ranks, positions = d["ranks"].astype(np.int64), d["positions"].astype(np.int64)
    assert bench.DUMP_SAMPLE // 2 < len(ranks) <= bench.DUMP_SAMPLE < want.num_suffixes
    assert (np.diff(ranks) > 0).all() and ranks[0] >= 0 and ranks[-1] < want.num_suffixes
    assert np.array_equal(d["sa"], want.sa[ranks].astype(np.float64))
    assert np.array_equal(d["lcp"], want.lcp[ranks].astype(np.float64))
    assert np.array_equal(d["text"], np.frombuffer(want.text, np.uint8)[positions].astype(np.float32))
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20


@pytest.mark.parametrize("bits", [32, 64])
def test_positions_above_2_31(S, bits):
    """2.3 Gbp: suffix positions that do not fit 31 bits, u32 and u64 results (what `sufr create` writes for a
    human genome is u32).  Checked with the size-independent sample check of the bench."""
    import torch
    import bench
    from sufr_b200 import _lib
    if torch.cuda.get_device_properties(0).total_memory < 120 * 2**30:
        pytest.skip("needs ~100 GB of device memory")
    text_len, starts = bench.record_layout(2_300_000_000)
    ctx = S.default_context(0)
    d = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    st = np.asarray(starts, dtype=np.uint64)
    assert _lib.lib().sufr_b200_synth_dna(ctx.handle, d.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                          ord("%")) == 0
    r = S.build(S.SufrBuilderArgs(text=b"", is_dna=True), index_bits=bits, ctx=ctx, result_memory=S.MEM_DEVICE,
                device_text=(d.data_ptr(), text_len))
    try:
        assert r.num_suffixes == text_len - 23
        v = r.verify()  # every pair, every position (positions >= 2^31 included)
        assert v["ok"] and v["pairs_checked"] == r.num_suffixes - 1, v
    finally:
        r.free()
        del d
        ctx.trim()
        torch.cuda.empty_cache()


@pytest.mark.parametrize("n", [10_000_000])
def test_config1_10mbp_random_dna(S, n):
    """BASELINE configs[0]: `sufr create --dna -n 16` on 10 Mbp random ACGT, u32 -- bit-exact vs the oracle."""
    rng = np.random.default_rng(1)
    text = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes() + b"$"
    want = O.oracle_build(text, is_dna=True, num_partitions=16, threads=16)
    got = S.build(S.SufrBuilderArgs(text=text, is_dna=True, num_partitions=16))
    assert got.num_suffixes == n + 1
    assert np.array_equal(got.sa, want.sa)
    assert np.array_equal(got.lcp, want.lcp)
    got.free()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_deep_repeats_fall_back_to_full_sort(S, world):
    """A shard cannot run prefix doubling on its own (it needs the rank of every position): the build is
    redone unsharded on each rank and the rank's slice is cut out.  Result still concatenates exactly."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = random.Random(world)
    text = rand_text(rng, 3000, b"ACGTN")[:-1] + b"ACGGT" * 1500 + rand_text(rng, 3000, b"ACGT")[:-1] + b"GT" * 2000 + b"$"
    for kw in (dict(is_dna=True), dict(is_dna=True, allow_ambiguity=True)):
        want = O.oracle_build(text, num_partitions=16, threads=4, **kw)
        shards = [S.build(S.SufrBuilderArgs(text=text, **kw), rank=r, world_size=world) for r in range(world)]
        assert any(s.c.doubling_rounds > 0 for s in shards)
        meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
        offs, total = shard_layout(meta)
        assert total == want.num_suffixes
        for r, s in enumerate(shards):
            s.set_shard_layout(offs[r], total)
            prev = previous_last_suffix(meta, r)
            if prev is not None and s.num_suffixes:
                s.patch_seam(prev)
        assert np.array_equal(np.concatenate([s.sa for s in shards]), want.sa)
        assert np.array_equal(np.concatenate([s.lcp for s in shards]), want.lcp)


def test_dense_active_set_uses_scan_compaction(S, monkeypatch):
    """Repetitive texts overflow the sparse append buffer of round 0; the ordered scan compaction takes over.
    (Forced here with a tiny buffer; the library reads the knob per build.)"""
    monkeypatch.setenv("SUFR_B200_DEBUG_SPARSE_CAP", "7")
    rng = random.Random(5)
    text = rand_text(rng, 40000, b"ACGT", repeat_p=0.2, max_rep=300)
    gpu_vs_oracle(S, text, is_dna=True)
    gpu_vs_oracle(S, text, seed_mask="111010010100110111")
    monkeypatch.delenv("SUFR_B200_DEBUG_SPARSE_CAP")
    gpu_vs_oracle(S, text, is_dna=True)


@pytest.mark.parametrize("name,size,kw", [
    ("config2b", 400_000, {}),
    ("config3", 300_000, dict(record_len=10_000)),
    ("config4", 500_000, {}),
    ("config5", 300_000, dict(max_unit=40, max_copies=300)),
])
def test_baseline_configs_small_vs_oracle(S, name, size, kw):
    """The BASELINE.json configs 2b-5 (generators: workloads.py) at sizes the oracle sorts in seconds."""
    import workloads
    w = workloads.ALL[name](size, **kw)
    flags = dict(w.flags)
    want = O.oracle_build(w.text, threads=8, sequence_starts=w.sequence_starts, sequence_names=w.sequence_names,
                          index_bits=w.index_bits, **flags)
    got = S.build(S.SufrBuilderArgs(text=w.text, sequence_starts=w.sequence_starts,
                                    sequence_names=w.sequence_names, **flags), index_bits=w.index_bits)
    assert got.text == want.text
    assert got.n_ranges == want.n_ranges
    if name == "config3":
        assert int(want.lcp.max()) < 32  # precondition: no two suffixes share Q residues
    assert np.array_equal(got.sa, want.sa)
    assert np.array_equal(got.lcp, want.lcp)
    # the size-independent checks used at full size agree with the oracle comparison
    sys_path_tools = str(__import__("conftest").ROOT / "tools")
    import sys
    sys.path.insert(0, sys_path_tools)
    from verify import check_pairs, check_positions
    ranks = np.random.default_rng(0).integers(0, got.num_suffixes, 500)
    assert check_pairs(got.text, got.sa, got.lcp, ranks, seed_mask=flags.get("seed_mask"),
                       max_query_len=flags.get("max_query_len"), n_ranges=got.n_ranges) == []
    assert check_positions(got.text, got.sa, is_dna=flags.get("is_dna", False),
                           allow_ambiguity=flags.get("allow_ambiguity", False))
    got.free()


def dna_with_rare(rng, n, rare=b"N%RYnacgt", rare_p=0.01, repeat_p=0.02, max_rep=200, runs=True):
    """DNA-like text: four dominant bytes plus rare irregular ones, repeats, and homopolymer runs (keys that
    are all zeros / all ones on the 2-bit fast path)."""
    out = bytearray()
    while len(out) < n:
        x = rng.random()
        if out and x < repeat_p:
            s = rng.randrange(len(out))
            out += out[s:s + rng.randrange(1, max_rep)]
        elif x < repeat_p + rare_p:
            out.append(rng.choice(rare))
        elif runs and x < repeat_p + rare_p + 0.002:
            out += bytes([rng.choice(b"AT")]) * rng.randrange(20, 120)
        else:
            out.append(rng.choice(b"ACGT"))
    return bytes(out[:n])


@pytest.mark.parametrize("flags", [dict(is_dna=True), dict(is_dna=True, ignore_softmask=True), dict(),
                                   dict(is_dna=True, allow_ambiguity=True)])
@pytest.mark.parametrize("deep", [False, True])
def test_fast2_device_u64_results_written_early(S, flags, deep, monkeypatch):
    """64-bit device results of the fast path are written by round 0 and patched where the refinement changes
    them; prefix doubling, the post-sort filter and the N-run rule fall back to the widening pass."""
    import torch
    rng = random.Random(seed_of("early_wide", str(flags), deep))
    text = dna_with_rare(rng, 120000) + (b"ACGGT" * 3000 if deep else b"") + b"$"
    want = O.oracle_build(text, threads=4, **flags)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    for env in (None, "1"):
        if env:
            monkeypatch.setenv("SUFR_B200_DEBUG_NO_EARLY_WIDE", env)
        r = S.build(S.SufrBuilderArgs(text=b"", **flags), index_bits=64, result_memory=S.MEM_DEVICE,
                    device_text=(d_text.data_ptr(), d_text.numel()))
        sa = r.sa_tensor().cpu().numpy().astype(np.uint64)
        lcp = r.lcp_tensor().cpu().numpy().astype(np.uint64)
        assert r.num_suffixes == want.num_suffixes
        assert np.array_equal(sa, want.sa.astype(np.uint64))
        assert np.array_equal(lcp, want.lcp.astype(np.uint64))
        r.free()


@pytest.mark.parametrize("world", [2, 5])
def test_fast2_sharded_device_u64_results(S, world):
    """The multi-GPU bench path: fast-path shards with 64-bit results left on the device, seams repaired there."""
    import torch
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = random.Random(seed_of("sharded_wide", world))
    text = dna_with_rare(rng, 200000) + b"$"
    want = O.oracle_build(text, is_dna=True, threads=4)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    shards = [S.build(S.SufrBuilderArgs(text=b"", is_dna=True), index_bits=64, result_memory=S.MEM_DEVICE,
                      device_text=(d_text.data_ptr(), d_text.numel()), rank=r, world_size=world) for r in range(world)]
    meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
    offs, total = shard_layout(meta)
    assert total == want.num_suffixes
    for r, s in enumerate(shards):
        s.set_shard_layout(offs[r], total)
        prev = previous_last_suffix(meta, r)
        if prev is not None and s.num_suffixes:
            s.patch_seam(prev)
    sa = np.concatenate([s.sa_tensor().cpu().numpy().astype(np.uint64) for s in shards if s.num_suffixes])
    lcp = np.concatenate([s.lcp_tensor().cpu().numpy().astype(np.uint64) for s in shards if s.num_suffixes])
    assert np.array_equal(sa, want.sa.astype(np.uint64))
    assert np.array_equal(lcp, want.lcp.astype(np.uint64))
    for s in shards:
        s.free()


@pytest.mark.parametrize("n", [5000, 70000, 300000])
@pytest.mark.parametrize("flags", [dict(is_dna=True), dict(is_dna=True, allow_ambiguity=True),
                                   dict(is_dna=True, ignore_softmask=True), dict()],
                         ids=["dna", "amb", "soft", "nodna"])
@pytest.mark.parametrize("tail", [b"$", b"", b"TTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTT"])
def test_fast2_path_matches_oracle(S, n, flags, tail, monkeypatch):
    """2-bit fast path of the first sort (DNA-like alphabets): irregular symbols become fill + exact ties."""
    rng = random.Random(seed_of(n, sorted(flags), tail))
    text = dna_with_rare(rng, n) + tail
    gpu_vs_oracle(S, text, **flags)
    # and the general 3-bit path gives the same answer
    monkeypatch.setenv("SUFR_B200_DEBUG_NO_FAST2", "1")
    gpu_vs_oracle(S, text, **flags)


def test_fast2_many_filtered_uses_compaction(S):
    rng = random.Random(17)
    text = dna_with_rare(rng, 120000, rare=b"N", rare_p=0.06) + b"$"
    gpu_vs_oracle(S, text, is_dna=True)


def test_fast2_symbols_above_t_and_below_a(S):
    rng = random.Random(23)
    text = dna_with_rare(rng, 90000, rare=b"#+BDHKVWXYZ[", rare_p=0.02) + b"$"
    gpu_vs_oracle(S, text)
    gpu_vs_oracle(S, text, is_dna=True, allow_ambiguity=True)


def test_fast2_deep_repeats_and_shards(S):
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = random.Random(29)
    text = dna_with_rare(rng, 40000) + b"ACGGT" * 3000 + dna_with_rare(rng, 20000) + b"T" * 5000 + b"$"
    _, _, doubling = gpu_vs_oracle(S, text, is_dna=True)
    assert doubling > 0
    want = O.oracle_build(text, is_dna=True, threads=4)
    for world in (2, 5):
        shards = [S.build(S.SufrBuilderArgs(text=text, is_dna=True), rank=r, world_size=world) for r in range(world)]
        meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
        for r, s in enumerate(shards):
            prev = previous_last_suffix(meta, r)
            if prev is not None and s.num_suffixes:
                s.patch_seam(prev)
        assert np.array_equal(np.concatenate([s.sa for s in shards]), want.sa)
        assert np.array_equal(np.concatenate([s.lcp for s in shards]), want.lcp)


@pytest.mark.parametrize("fuse", ["1", "0"])
@pytest.mark.parametrize("kw", [dict(is_dna=True), dict(is_dna=True, allow_ambiguity=True), dict()],
                         ids=["filtered", "ambiguity", "bytes"])
def test_shard_selection_fused_with_first_radix_pass(S, monkeypatch, fuse, kw):
    """Key-range shards select their records and sort them in four passes; the variant that generates them already in
    first-digit order (selection fused with key generation and the first radix pass, SUFR_B200_DEBUG_SHARD_FUSE=1:
    measured, not the default) must give the same arrays.  Both ways for 2, 3, 8 and 33 shards (some of them empty)."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    monkeypatch.setenv("SUFR_B200_DEBUG_SHARD_FUSE", fuse)
    rng = random.Random(len(kw) + int(fuse))
    text = dna_with_rare(rng, 90000) + b"ACGT" * 300 + rand_text(rng, 20000, b"ACGT", repeat_p=0.05, max_rep=200)[:-1] + b"$"
    want = O.oracle_build(text, threads=4, **kw)
    for world in (2, 3, 8, 33):
        shards = [S.build(S.SufrBuilderArgs(text=text, **kw), rank=r, world_size=world) for r in range(world)]
        meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
        offs, total = shard_layout(meta)
        assert total == want.num_suffixes
        for r, sh in enumerate(shards):
            sh.set_shard_layout(offs[r], total)
            prev = previous_last_suffix(meta, r)
            if prev is not None and sh.num_suffixes:
                sh.patch_seam(prev)
        assert np.array_equal(np.concatenate([sh.sa for sh in shards]), want.sa)
        assert np.array_equal(np.concatenate([sh.lcp for sh in shards]), want.lcp)
        for sh in shards:
            sh.free()


def family_text(rng, n, seg_len=2000, copies=30, mut=0.01):
    """Random DNA with one segment copied `copies` times, each copy with ~1 % substitutions: suffix groups of up to
    `copies` members whose common prefixes run to hundreds of bases (a repeat family of a genome)."""
    acgt = b"ACGT"
    seg = bytes(rng.choice(acgt) for _ in range(seg_len))
    out = bytearray()
    per = (n - copies * seg_len) // copies
    nrng = np.random.default_rng(rng.randrange(1 << 30))
    for _ in range(copies):
        out += np.frombuffer(acgt, dtype=np.uint8)[nrng.integers(0, 4, per)].tobytes()
        c = bytearray(seg)
        for i in range(seg_len):
            if rng.random() < mut:
                c[i] = rng.choice(acgt)
        out += c
    return bytes(out) + b"$"


@pytest.mark.parametrize("block_tail", [True, False])
def test_repeat_families_finish_by_direct_comparison(S, monkeypatch, block_tail):
    """Subset attempts (shards, pre-filtered builds) cannot run prefix doubling: the deep tail -- pairs and small groups
    by one thread each, families of up to 8192 members by one block each (bitonic network over direct suffix
    comparisons) -- is finished in one step instead of one word round per 21 bases."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    if not block_tail:
        monkeypatch.setenv("SUFR_B200_DEBUG_NO_BLOCK_TAIL", "1")
    rng = random.Random(77)
    text = family_text(rng, 4_000_000)   # the family is 1.5 % of the text: the tail starts right after the third word
    want = O.oracle_build(text, is_dna=True, threads=4)
    rounds = []
    for world in (1, 2, 3):
        shards = [S.build(S.SufrBuilderArgs(text=text, is_dna=True), rank=r, world_size=world) for r in range(world)]
        if world > 1:
            assert all(sh.c.doubling_rounds == 0 for sh in shards)
            rounds.append(max(sh.c.refine_rounds for sh in shards))
        meta = [(sh.num_suffixes, sh.first_suffix, sh.last_suffix) for sh in shards]
        offs, total = shard_layout(meta)
        assert total == want.num_suffixes
        for r, sh in enumerate(shards):
            sh.set_shard_layout(offs[r], total)
            prev = previous_last_suffix(meta, r)
            if prev is not None and sh.num_suffixes:
                sh.patch_seam(prev)
        assert np.array_equal(np.concatenate([sh.sa for sh in shards]), want.sa)
        assert np.array_equal(np.concatenate([sh.lcp for sh in shards]), want.lcp)
        for sh in shards:
            sh.free()
    if block_tail:
        assert max(rounds) <= 8, rounds      # the tail starts after the third word
    else:
        assert max(rounds) >= 12, rounds     # one round per key word until the families have split up otherwise


def test_sharded_build_writes_one_file(S, tmp_path):
    """Every rank pwrites its slice into the same `.sufr` (sufr_b200_write, sharded): byte-identical to the
    single-process file."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = random.Random(31)
    text = dna_with_rare(rng, 150000) + b"$"
    single = tmp_path / "single.sufr"
    S.SufrBuilder(S.SufrBuilderArgs(text=text, path=str(single), is_dna=True, sequence_names=["x"]), 32)
    out = tmp_path / "sharded.sufr"
    world = 4
    args = S.SufrBuilderArgs(text=text, path=str(out), is_dna=True, sequence_names=["x"])
    shards = [S.build(args, rank=r, world_size=world) for r in range(world)]
    meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
    offs, total = shard_layout(meta)
    for r, s in enumerate(shards):
        s.set_shard_layout(offs[r], total)
        prev = previous_last_suffix(meta, r)
        if prev is not None and s.num_suffixes:
            s.patch_seam(prev)
        s.write()
    assert out.read_bytes() == single.read_bytes()


@pytest.mark.parametrize("golden,fasta,flags", [c for c in GOLDEN_CASES if c[0] in
                                                ("1.sufr", "2d.sufr", "2ns.sufr", "long_dna_sequence_allow_ambiguity.sufr",
                                                 "uniprot-masked.sufr", "abba.sufr")], ids=lambda v: v if isinstance(v, str) else "")
def test_cli_create_writes_golden_files(tmp_path, golden, fasta, flags):
    """`sufr-b200 create` with the reference's flags (sufr/tests/cli.rs:55-302) -> byte-identical `.sufr`."""
    import subprocess
    exe = __import__("conftest").ROOT / "sufr_b200" / "sufr-b200"
    out = tmp_path / golden
    cmd = [str(exe), "create", "-o", str(out), str(GOLDEN / "inputs" / fasta)]
    if flags.get("is_dna"):
        cmd.append("--dna")
    if flags.get("allow_ambiguity"):
        cmd.append("--allow-ambiguity")
    if flags.get("ignore_softmask"):
        cmd.append("--ignore-softmask")
    if "delimiter" in flags:
        cmd += ["--sequence-delimiter", flags["delimiter"].decode()]
    if "seed_mask" in flags:
        cmd += ["--seed-mask", flags["seed_mask"]]
    r = subprocess.run(cmd + ["--log", "info"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Sorted" in r.stdout
    assert out.read_bytes() == (GOLDEN / "expected" / golden).read_bytes()


def test_filter_after_full_sort_fast_and_generic_paths(S, monkeypatch):
    """Repetitive DNA with scattered N: the filtered attempt gives up, everything is sorted with prefix
    doubling, and the non-indexed suffixes are dropped afterwards -- by the look-back kernel, and (forced)
    by the generic segmented-min scan.  A long N run overflows the look-back and takes the scan by itself."""
    rng = random.Random(37)
    base = dna_with_rare(rng, 60000, rare=b"N", rare_p=0.01, repeat_p=0.0)
    text = base + base[:30000] + base[10000:50000] + b"$"      # long exact repeats => doubling
    _, _, doubling = gpu_vs_oracle(S, text, is_dna=True)
    assert doubling > 0
    monkeypatch.setenv("SUFR_B200_DEBUG_SLOW_FILTER", "1")
    gpu_vs_oracle(S, text, is_dna=True)
    monkeypatch.delenv("SUFR_B200_DEBUG_SLOW_FILTER")
    text2 = base[:20000] + b"N" * 3000 + base[:20000] + b"N" * 700 + base[5000:15000] + b"$"
    gpu_vs_oracle(S, text2, is_dna=True)


def test_sharded_fallback_on_some_ranks_only(S):
    """Found by tools/stress.py: when only SOME ranks hit deep repeats (long N runs under --allow-ambiguity)
    and redo their build unsharded, they must keep the key-range cuts every rank derived first."""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = np.random.default_rng(11)
    t = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 120000)].copy()
    t[30000:32200] = ord("N")
    t[90000:91001] = ord("N")
    text = t.tobytes() + b"$"
    for flags in (dict(is_dna=True, allow_ambiguity=True), dict(is_dna=True, allow_ambiguity=True, ignore_softmask=True)):
        want = O.oracle_build(text, threads=4, **flags)
        for world in (2, 3, 5):
            shards = [S.build(S.SufrBuilderArgs(text=text, **flags), rank=r, world_size=world) for r in range(world)]
            meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
            offs, total = shard_layout(meta)
            assert total == want.num_suffixes
            for r, s in enumerate(shards):
                s.set_shard_layout(offs[r], total)
                prev = previous_last_suffix(meta, r)
                if prev is not None and s.num_suffixes:
                    s.patch_seam(prev)
            assert np.array_equal(np.concatenate([s.sa for s in shards]), want.sa)
            assert np.array_equal(np.concatenate([s.lcp for s in shards]), want.lcp)


def test_sharded_host_results_from_device_text(S):
    """bench.py's multi-GPU e2e path: the text is in device memory, results go to the host, ranks > 0 carry no
    transformed text -- the seam repair reads windows of the caller's device text."""
    import torch
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    rng = random.Random(41)
    text = dna_with_rare(rng, 100000, rare=b"nacgt%", rare_p=0.02) + b"$"
    want = O.oracle_build(text, is_dna=True, threads=4)
    d = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    world = 3
    shards = [S.build(S.SufrBuilderArgs(text=b"", is_dna=True), rank=r, world_size=world,
                      device_text=(d.data_ptr(), d.numel())) for r in range(world)]
    meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
    offs, total = shard_layout(meta)
    for r, s in enumerate(shards):
        s.set_shard_layout(offs[r], total)
        prev = previous_last_suffix(meta, r)
        if prev is not None and s.num_suffixes:
            s.patch_seam(prev)
    assert shards[0].text == want.text
    assert np.array_equal(np.concatenate([s.sa for s in shards]), want.sa)
    assert np.array_equal(np.concatenate([s.lcp for s in shards]), want.lcp)


@pytest.mark.parametrize("bits", [32, 64])
def test_compact_host_transfer(S, bits, monkeypatch):
    """Large host results travel as LCP bytes + exceptions (and u32 SA for u64 output) and are widened on the
    host; forced on for a small input here, with LCP values on both sides of the byte limit."""
    monkeypatch.setenv("SUFR_B200_DEBUG_COMPACT_MIN", "1")
    rng = random.Random(43)
    base = dna_with_rare(rng, 60000, rare=b"N", rare_p=0.002)
    text = base + base[1000:1400] + base[5000:5254] + base[9000:9256] + b"$"   # LCPs of 400, 254, 256
    gpu_vs_oracle(S, text, index_bits=bits, is_dna=True)
    gpu_vs_oracle(S, text, index_bits=bits)
    # a text whose LCP values mostly exceed a byte falls back to the plain transfer
    gpu_vs_oracle(S, b"ACGT" * 3000 + b"$", index_bits=bits, is_dna=True)
