"""CPU-only tests of the host side of the product: the C ABI surface, the SeedMask / FASTA / `.sufr`
writer code in libsufr_b200.so, and the multi-rank host logic (gloo, world_size 2).  No CUDA compute."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES, ROOT
import oracle as O
from sufrfile import parse_sufr


@pytest.fixture(scope="module")
def S():
    subprocess.check_call(["make", "-C", str(ROOT / "sufr_b200" / "csrc"), "-s", "-j8"])
    import sufr_b200
    return sufr_b200


def test_library_exports_every_declared_symbol(S):
    from sufr_b200 import _lib
    header = (ROOT / "include" / "sufr_b200.h").read_text()
    declared = sorted(set(re.findall(r"\b(sufr_b200_[a-z0-9_]+)\s*\(", header)))
    assert declared == sorted(_lib.ABI_SYMBOLS)
    L = _lib.lib()
    for sym in declared:
        assert getattr(L, sym) is not None
    assert L.sufr_b200_abi_version() == 2
    out = subprocess.check_output(["nm", "-D", "--defined-only", str(_lib.LIB_PATH)], text=True)
    exported = set(re.findall(r" T (sufr_b200_[a-z0-9_]+)", out))
    assert set(declared) <= exported


def test_struct_layouts_match_header(S):
    """ctypes mirrors vs. the C compiler's layout of the header structs."""
    from sufr_b200 import _lib
    src = r'''
    #include "sufr_b200.h"
    #include <stdio.h>
    #include <stddef.h>
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu\n", sizeof(SufrB200Args), sizeof(SufrB200Result), sizeof(SufrB200Timings),
             sizeof(SufrB200Sequences), sizeof(SufrB200VerifyReport), offsetof(SufrB200VerifyReport, ms));
      printf("%zu %zu %zu %zu %zu\n", offsetof(SufrB200Args, max_query_len), offsetof(SufrB200Args, seed_mask),
             offsetof(SufrB200Args, rank), offsetof(SufrB200Result, timings), offsetof(SufrB200Result, owner));
      return 0; }'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", str(ROOT / "include"), "-o", os.path.join(d, "t"), os.path.join(d, "t.c")])
        out = subprocess.check_output([os.path.join(d, "t")], text=True).split()
    sizes = [C.sizeof(_lib.Args), C.sizeof(_lib.Result), C.sizeof(_lib.Timings), C.sizeof(_lib.Sequences),
             C.sizeof(_lib.VerifyReport), _lib.VerifyReport.ms.offset]
    offs = [_lib.Args.max_query_len.offset, _lib.Args.seed_mask.offset, _lib.Args.rank.offset,
            _lib.Result.timings.offset, _lib.Result.owner.offset]
    assert [int(x) for x in out] == sizes + offs


def test_no_cuda_device_fails_loudly(S):
    """No CPU fallback: without a GPU every compute entry point errors."""
    from sufr_b200 import _lib
    if _lib.lib().sufr_b200_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(S.SufrError, match="no CUDA device"):
        S.SufrBuilder(S.SufrBuilderArgs(text=b"ACGT$"))


def test_product_does_not_reference_the_oracle():
    for path in list((ROOT / "sufr_b200").rglob("*")) + [ROOT / "include" / "sufr_b200.h"]:
        if path.suffix in (".py", ".cu", ".cuh", ".cpp", ".hpp", ".h") or path.name == "Makefile":
            text = path.read_text()
            for needle in ("libsufr_oracle", "sufr_oracle", "import oracle", "from oracle", "oracle/"):
                hits = [ln for ln in text.splitlines() if needle in ln and "never" not in ln and "no " not in ln.lower()
                        and "not " not in ln.lower() and "nothing" not in ln.lower()]
                assert not hits, (path, hits)


def test_seed_mask_mirror(S):
    # types.rs:62-78, 634-737
    for bad in ["", "0", "01", "10", "11", "0101", "1010", "1021", "1111", "abc", "1", "111", "00", "0111",
                "11100", "1a01"]:
        assert not S.SeedMask.is_valid(bad)
        with pytest.raises(S.SufrError, match="Invalid seed mask"):
            S.SeedMask.new(bad)
    m = S.SeedMask.new("110110101")
    assert (m.bytes, m.positions, m.differences, m.weight) == \
        ([1, 1, 0, 1, 1, 0, 1, 0, 1], [0, 1, 3, 4, 6, 8], [0, 0, 1, 1, 2, 3], 6)
    m = S.SeedMask.new("11101101101000011")
    assert m.positions == [0, 1, 2, 4, 5, 7, 8, 10, 15, 16] and m.differences == [0, 0, 0, 1, 1, 2, 2, 3, 7, 7]
    assert str(m) == "11101101101000011"
    for mask in ["101", "1001", "1101", "10101", "1110110110100001", "10111011", "111010010100110111"]:
        assert S.SeedMask.is_valid(mask)
        want = O.seed_mask(mask)
        got = S.SeedMask.new(mask)
        assert (got.bytes, got.positions, got.differences, got.weight) == want


def test_find_lcp_full_offset_mirror(S):
    # util.rs:289-314, plus agreement with the oracle on more masks
    assert [S.find_lcp_full_offset(i, "101") for i in range(3)] == [0, 2, 3]
    assert [S.find_lcp_full_offset(i, "11011") for i in range(5)] == [0, 1, 3, 4, 5]
    assert [S.find_lcp_full_offset(i, "10011001") for i in range(5)] == [0, 3, 4, 7, 8]
    assert S.find_lcp_full_offset(17, None) == 17
    for mask in ["1101101101", "111010010100110111", "10111011"]:
        w = mask.count("1")
        for l in range(w + 1):
            assert S.find_lcp_full_offset(l, mask) == O.find_lcp_full_offset(l, mask)


@pytest.mark.parametrize("fasta", ["1.fa", "2.fa", "3.fa", "abba.fa", "long_dna_sequence.fa", "smol.fa", "uniprot.fa"])
@pytest.mark.parametrize("delim", [b"%", b"N"])
def test_read_sequence_file_matches_oracle(S, fasta, delim):
    a = S.read_sequence_file(GOLDEN / "inputs" / fasta, delim)
    b = O.read_sequence_file(GOLDEN / "inputs" / fasta, delim)
    assert (a.seq, a.start_positions, a.sequence_names) == (b.seq, b.start_positions, b.sequence_names)


def test_read_sequence_file_kat_and_errors(S, tmp_path):
    d = S.read_sequence_file(GOLDEN / "inputs" / "2.fa", b"N")  # util.rs:183-194
    assert (d.seq, d.start_positions, d.sequence_names) == (b"ACGTacgtNacgtACGT$", [0, 9], ["ABC", "DEF"])
    with pytest.raises(S.SufrError):
        S.read_sequence_file(GOLDEN / "inputs" / "empty.fa")
    with pytest.raises(S.SufrError):
        S.read_sequence_file(tmp_path / "missing.fa")
    fq = tmp_path / "x.fq"
    fq.write_text("@r1 desc\nACGT\n+\nIIII\n@r2\nGGCC\n+\nIIII\n")
    d = S.read_sequence_file(fq)
    assert (d.seq, d.start_positions, d.sequence_names) == (b"ACGT%GGCC$", [0, 5], ["r1", "r2"])
    crlf = tmp_path / "crlf.fa"
    crlf.write_bytes(b">a b\r\nAC\r\nGT\r\n>c\r\nTT\r\n")
    d = S.read_sequence_file(crlf)
    assert (d.seq, d.start_positions, d.sequence_names) == (b"ACGT%TT$", [0, 5], ["a", "c"])


@pytest.mark.parametrize("seed,records,crlf,final_newline", [(1, 3, False, True), (2, 2000, True, False),
                                                             (3, 40, False, False)])
def test_parallel_fasta_ingest_matches_serial_restatement(S, tmp_path, seed, records, crlf, final_newline):
    """Files of tens of MB are read and parsed by several threads (slices cut at line starts): same text,
    starts and names as the serial restatement of util.rs:51-89, whatever the line structure."""
    import random
    rng = random.Random(seed)
    total = 40_000_000
    eol = b"\r\n" if crlf else b"\n"
    parts = []
    for r in range(records):
        parts.append(b">rec%d some description" % r + eol)
        left = total // records
        body = bytes(rng.choices(b"ACGTN", k=1000)) * (left // 1000 + 1)
        pos = 0
        while pos < left:
            w = rng.choice([60, 61, 80, 1, 200, 100000])
            parts.append(body[pos:pos + min(w, left - pos)] + eol)
            pos += w
            if rng.random() < 0.01:
                parts.append(eol)  # blank line inside a record
    blob = b"".join(parts)
    if not final_newline:
        blob = blob.rstrip(b"\r\n")
    fa = tmp_path / "big.fa"
    fa.write_bytes(blob)
    a = S.read_sequence_file(fa, b"%")
    b = O.read_sequence_file(fa, b"%")
    assert a.start_positions == b.start_positions
    assert a.sequence_names == b.sequence_names
    assert a.seq == b.seq


@pytest.mark.parametrize("codec", ["gz", "gz_multi_member", "bz2", "xz", "zst"])
def test_compressed_input(S, tmp_path, codec):
    """needletail decompresses gz / bz2 / xz / zstd transparently (util.rs:55); so does read_sequence_file here."""
    import bz2, gzip, lzma, random
    rng = random.Random(5)
    fa = tmp_path / "t.fa"
    with open(fa, "w") as f:
        for r in range(300):
            f.write(f">seq{r} description\n")
            body = "".join(rng.choice("ACGTN") for _ in range(rng.randrange(1, 5000)))
            for i in range(0, len(body), 70):
                f.write(body[i:i + 70] + "\n")
    raw = fa.read_bytes()
    if codec == "gz":
        blob = gzip.compress(raw)
    elif codec == "gz_multi_member":  # what bgzip and `cat a.gz b.gz` produce
        blob = gzip.compress(raw[:len(raw) // 3]) + gzip.compress(raw[len(raw) // 3:])
    elif codec == "bz2":
        blob = bz2.compress(raw)
    elif codec == "xz":
        blob = lzma.compress(raw)
    else:
        pa = pytest.importorskip("pyarrow")
        blob = pa.compress(raw, codec="zstd", asbytes=True)
    packed = tmp_path / f"t.fa.{codec}"
    packed.write_bytes(blob)
    want = O.read_sequence_file(fa, b"%")
    got = S.read_sequence_file(packed, b"%")
    assert (got.seq, got.start_positions, got.sequence_names) == (want.seq, want.start_positions, want.sequence_names)
    packed.write_bytes(blob[:len(blob) // 2])
    with pytest.raises(S.SufrError, match="truncated|corrupt"):
        S.read_sequence_file(packed, b"%")


@pytest.mark.parametrize("crlf", [False, True])
def test_parallel_fastq_ingest_matches_serial_restatement(S, tmp_path, crlf):
    """FASTQ is parsed by several threads too: a slice starts at an '@' line whose second successor is a '+' line --
    qualities that begin with '@' or '+' must not confuse it."""
    import random
    rng = random.Random(11)
    eol = "\r\n" if crlf else "\n"
    fq = tmp_path / "big.fq"
    with open(fq, "w", newline="") as f:
        for r in range(150_000):
            seq = "".join(rng.choice("ACGTN") for _ in range(rng.randrange(20, 150)))
            qual = "".join(rng.choice("@+IJ#5") for _ in range(len(seq)))
            f.write(f"@read{r} extra{eol}{seq}{eol}+{eol}{qual}{eol}")
    assert fq.stat().st_size > 20_000_000  # several slices
    want = O.read_sequence_file(fq, b"%")
    got = S.read_sequence_file(fq, b"%")
    assert got.start_positions == want.start_positions
    assert got.sequence_names == want.sequence_names
    assert got.seq == want.seq


def test_create_rejects_sharded_arguments(S):
    from sufr_b200 import _lib
    import ctypes as C
    args = _lib.Args()
    args.world_size = 2
    args.rank = 1
    rc = _lib.lib().sufr_b200_create(C.byref(args), 0, None)
    assert rc == _lib.ERR_ARGUMENT
    assert b"single-process" in _lib.lib().sufr_b200_last_error()


def _host_result(S, o, shard=None):
    """A SufrB200Result in host memory filled from oracle arrays (exercises the writer without a GPU)."""
    from sufr_b200 import _lib
    r = _lib.Result()
    bits = o.index_bits
    lo, hi = (0, o.num_suffixes) if shard is None else shard
    keep = dict(text=np.frombuffer(o.text, np.uint8).copy(), sa=o.sa[lo:hi].copy(), lcp=o.lcp[lo:hi].copy())
    r.index_bits, r.memory, r.text_len = bits, _lib.MEM_HOST, len(o.text)
    r.num_suffixes, r.total_suffixes, r.shard_offset = hi - lo, o.num_suffixes, lo
    r.text = keep["text"].ctypes.data
    r.sa = keep["sa"].ctypes.data
    r.lcp = keep["lcp"].ctypes.data
    return r, keep


@pytest.mark.parametrize("golden,fasta,flags", GOLDEN_CASES, ids=[c[0] for c in GOLDEN_CASES])
@pytest.mark.parametrize("world", [1, 3])
def test_sufr_writer_matches_golden_bytes(S, tmp_path, golden, fasta, flags, world):
    """sufr_b200_write (single shard, and three ranks pwriting into one file) == the reference's file."""
    from sufr_b200 import _lib
    from sufr_b200.builder import _CArgs
    flags = dict(flags)
    delim = flags.pop("delimiter", b"%")
    seq = S.read_sequence_file(GOLDEN / "inputs" / fasta, delim)
    o = O.oracle_build(seq.seq, sequence_starts=seq.start_positions, sequence_names=seq.sequence_names, **flags)
    out = tmp_path / "out.sufr"
    out.write_bytes(b"stale" * 300000)  # an older, longer file must not leak through
    args = S.SufrBuilderArgs(text=seq.seq, path=str(out), sequence_starts=seq.start_positions,
                             sequence_names=seq.sequence_names, **flags)
    s = o.num_suffixes
    cuts = [s * r // world for r in range(world + 1)]
    for rank in reversed(range(world)):  # any order works: offsets are absolute
        c = _CArgs(args, rank=rank, world_size=world)
        r, keep = _host_result(S, o, (cuts[rank], cuts[rank + 1]))
        assert _lib.lib().sufr_b200_write(C.byref(c.c), C.byref(r)) == 0, _lib.lib().sufr_b200_last_error()
    assert out.read_bytes() == (GOLDEN / "expected" / golden).read_bytes()


def test_writer_sections_written_by_several_threads(S, tmp_path, monkeypatch):
    """Large sections are cut into pieces that several threads pwrite; forced on a small file here."""
    from sufr_b200 import _lib
    from sufr_b200.builder import _CArgs
    monkeypatch.setenv("SUFR_B200_DEBUG_WRITE_PIECE", "1000")
    seq = S.read_sequence_file(GOLDEN / "inputs" / "uniprot.fa", b"%")
    o = O.oracle_build(seq.seq, sequence_starts=seq.start_positions, sequence_names=seq.sequence_names)
    out = tmp_path / "out.sufr"
    args = S.SufrBuilderArgs(text=seq.seq, path=str(out), sequence_starts=seq.start_positions,
                             sequence_names=seq.sequence_names)
    r, keep = _host_result(S, o)
    c = _CArgs(args)
    assert _lib.lib().sufr_b200_write(C.byref(c.c), C.byref(r)) == 0
    assert out.read_bytes() == (GOLDEN / "expected" / "uniprot.sufr").read_bytes()


def test_writer_u64_layout(S, tmp_path):
    from sufr_b200 import _lib
    from sufr_b200.builder import _CArgs
    o = O.oracle_build(b"ACGTNNACGT$", is_dna=True, allow_ambiguity=True, index_bits=64, num_partitions=2)
    out = tmp_path / "u64.sufr"
    args = S.SufrBuilderArgs(text=b"ACGTNNACGT$", path=str(out), is_dna=True, allow_ambiguity=True)
    c = _CArgs(args)
    r, keep = _host_result(S, o)
    assert _lib.lib().sufr_b200_write(C.byref(c.c), C.byref(r)) == 0
    assert out.read_bytes() == o.file_bytes


def test_writer_io_error_message(S, tmp_path):
    from sufr_b200 import _lib
    from sufr_b200.builder import _CArgs
    o = O.oracle_build(b"ACGT$", is_dna=True)
    bad = tmp_path / "no_such_dir" / "x.sufr"
    c = _CArgs(S.SufrBuilderArgs(text=b"ACGT$", path=str(bad), is_dna=True))
    r, keep = _host_result(S, o)
    assert _lib.lib().sufr_b200_write(C.byref(c.c), C.byref(r)) == _lib.ERR_IO
    msg = _lib.lib().sufr_b200_last_error().decode()
    assert msg.startswith(f"{bad}: ")  # "{filename}: {io error}", sufr_builder.rs:820


def test_cli_flag_surface(S):
    """`sufr-b200 create` mirrors the reference's clap definitions (sufr/src/lib.rs:85-125)."""
    exe = ROOT / "sufr_b200" / "sufr-b200"
    help_text = subprocess.run([str(exe), "create", "--help"], capture_output=True, text=True).stdout
    for flag in ["--num-partitions", "--max-query-len", "--output", "--dna", "--allow-ambiguity", "--ignore-softmask",
                 "--sequence-delimiter", "--seed-mask", "--random-seed", "[default: 16]", "[default: %]", "[default: 42]"]:
        assert flag in help_text
    r = subprocess.run([str(exe), "create", "-m", "3", "-s", "101", "x.fa"], capture_output=True, text=True)
    assert r.returncode == 2 and "cannot be used with" in r.stderr      # clap conflicts_with, lib.rs:95
    r = subprocess.run([str(exe), "create"], capture_output=True, text=True)
    assert r.returncode == 2
    r = subprocess.run([str(exe), "create", str(GOLDEN / "inputs" / "empty.fa")], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith("Error: ")        # cli.rs:102-109 create_empty_dies


def test_bench_reference_arm_dump_outputs(tmp_path):
    """`bench.py --impl reference --dump-outputs` (CPU only): the last timed step's arrays, whole below
    bench.DUMP_SAMPLE, and --steps sets the number of timed steps."""
    import json
    import bench
    bases = 300_000
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--bases", str(bases),
                        "--cpu-sample", str(bases), "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
    text_len, starts = bench.record_layout(bases)
    text = bench.synth_prefix_numpy(bases, text_len, starts)[:-1] + b"$"  # the arm's prefix of the workload text
    want = O.oracle_build(text, is_dna=True, index_bits=64)
    d = {f.stem: np.load(f) for f in tmp_path.glob("*.npy")}
    assert d["sizes"].tolist() == [want.num_suffixes, len(text)]
    assert d["ranks"].tolist() == list(range(want.num_suffixes))
    assert np.array_equal(d["sa"], want.sa.astype(np.float64))
    assert np.array_equal(d["lcp"], want.lcp.astype(np.float64))
    assert np.array_equal(d["text"], np.frombuffer(text, np.uint8).astype(np.float32))


def test_distributed_meta_logic():
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    meta = [(0, 0, 0), (5, 10, 11), (0, 0, 0), (7, 3, 4), (2, 8, 9)]
    assert [previous_last_suffix(meta, r) for r in range(5)] == [None, None, 11, 11, 4]
    assert shard_layout(meta) == ([0, 0, 5, 5, 12], 14)


GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from sufr_b200.distributed import finish_shard, gather_meta, previous_last_suffix, shard_layout
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
mine = [(4, 100, 101), (6, 200, 201)][rank]
meta = gather_meta(*mine)
assert meta == [(4, 100, 101), (6, 200, 201)], meta
offs, total = shard_layout(meta)
assert (offs, total) == ([0, 4], 10)
assert previous_last_suffix(meta, rank) == (None if rank == 0 else 101)


class FakeShard:  # what finish_shard needs from a BuildResult
    def __init__(self, n, first, last):
        self.num_suffixes, self.first_suffix, self.last_suffix = n, first, last
        self.layout, self.seam = None, None
    def set_shard_layout(self, off, tot):
        self.layout = (off, tot)
    def patch_seam(self, prev):
        self.seam = prev


shard = FakeShard(*mine)
finish_shard(shard)
assert shard.layout == ((0, 10) if rank == 0 else (4, 10)), shard.layout
assert shard.seam == (None if rank == 0 else 101), shard.seam
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
'''


def test_distributed_gloo_world2(tmp_path):
    """N>1 host logic under torch.distributed (gloo, 2 processes, CPU)."""
    import socket
    script = tmp_path / "w.py"
    script.write_text(GLOO_WORKER)
    with socket.socket() as s:  # a free port: a fixed one collides with another run on the same host
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), str(ROOT)], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
