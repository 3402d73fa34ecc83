"""The full on-device verifier (sufr_b200_verify): it accepts results that are bit-exact with the oracle, in every
mode, and it catches corrupted suffix / LCP arrays.  Also the large oracle comparisons (>= 100 M suffixes)."""
import random
import zlib

import numpy as np
import pytest

import oracle as O
import workloads

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S():
    import sufr_b200
    return sufr_b200


def device_build(S, text, index_bits=32, **kw):
    import torch
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    args = S.SufrBuilderArgs(text=b"", **kw)
    r = S.build(args, index_bits=index_bits, result_memory=S.MEM_DEVICE, device_text=(t.data_ptr(), t.numel()))
    r._keep = t
    return r


def seed_of(*parts) -> int:
    """Deterministic seed (Python's hash() of str is randomised per process)."""
    return zlib.crc32(repr(parts).encode()) & 0xFFFF


def rand_dna(seed, n, repeat_p=0.0, max_rep=60, alphabet=b"ACGT"):
    rng = random.Random(seed)
    out = bytearray()
    while len(out) < n:
        if out and rng.random() < repeat_p:
            s = rng.randrange(len(out))
            out += out[s:s + rng.randrange(1, max_rep)]
        else:
            out.append(rng.choice(alphabet))
    return bytes(out[:n]) + b"$"


MODES = {
    "dna": dict(is_dna=True),
    "dna_amb": dict(is_dna=True, allow_ambiguity=True),
    "dna_amb_soft": dict(is_dna=True, allow_ambiguity=True, ignore_softmask=True),
    "protein": dict(),
    "mask": dict(is_dna=True, seed_mask="1101101101"),
    "mql": dict(max_query_len=12),
}


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("bits", [32, 64])
def test_verifier_accepts_oracle_exact_results(S, mode, bits):
    kw = MODES[mode]
    alphabet = b"ACGTNacgtn%" if kw.get("is_dna") else b"ACDEFGHIKLMNPQRSTVWY%"
    text = rand_dna(seed_of(mode, bits), 60_000, repeat_p=0.02, alphabet=alphabet)
    want = O.oracle_build(text, num_partitions=8, threads=4, index_bits=bits, **kw)
    r = device_build(S, text, bits, **kw)
    try:
        rep = r.verify()
        if mode != "mql":  # with ties under --max-query-len the reference itself is schedule dependent (DESIGN 3.4)
            assert np.array_equal(r.sa_tensor().cpu().numpy().astype(want.sa.dtype), want.sa)
            assert np.array_equal(r.lcp_tensor().cpu().numpy().astype(want.lcp.dtype), want.lcp)
        assert rep["ok"], rep
        assert rep["pairs_checked"] == r.num_suffixes - 1
        assert rep["expected_suffixes"] == want.num_suffixes
        assert rep["max_lcp"] == int(r.lcp_tensor().max().item())
    finally:
        r.free()


def test_verifier_catches_corruption(S):
    text = rand_dna(5, 200_000, repeat_p=0.01)
    for what in ("swap", "lcp", "dup", "range"):
        r = device_build(S, text, 32, is_dna=True)
        try:
            assert r.verify()["ok"]
            sa, lcp = r.sa_tensor(), r.lcp_tensor()
            j = 123_456
            if what == "swap":
                a, b = sa[j].item(), sa[j + 1].item()
                sa[j], sa[j + 1] = b, a
            elif what == "lcp":
                lcp[j] += 1
            elif what == "dup":
                sa[j] = sa[j + 7]
            else:
                sa[j] = len(text) + 5
            rep = r.verify()
            assert not rep["ok"], (what, rep)
            if what == "swap":
                assert rep["order_errors"] >= 1
            if what == "lcp":
                assert rep["lcp_errors"] == 1 and rep["first_bad_rank"] == j
            if what == "dup":
                assert rep["duplicates"] >= 1
            if what == "range":
                assert rep["out_of_range"] == 1
        finally:
            r.free()


def tandem_text(seed, n):
    """Deep repeats: tandem arrays with units of 1-40 bp, a few long N runs (>= 1000) after different bases."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    parts, size, k = [], 0, 0
    while size < n:
        k += 1
        if k % 7 == 0:
            seg = np.full(int(rng.integers(1000, 3000)), ord("N"), dtype=np.uint8)
        elif k % 2:
            seg = np.tile(acgt[rng.integers(0, 4, int(rng.integers(1, 41)))], int(rng.integers(50, 3000)))
        else:
            seg = acgt[rng.integers(0, 4, int(rng.integers(500, 5000)))]
        parts.append(seg)
        size += len(seg)
    return np.concatenate(parts)[:n].tobytes() + b"A$"


@pytest.mark.parametrize("kw", [dict(is_dna=True, allow_ambiguity=True), dict(is_dna=True), dict()],
                         ids=["linear_time_proof", "filtered_direct", "bytes"])
def test_verifier_on_deep_repeats(S, kw):
    """LCP values far above the per-pair budget: deferred pairs are settled by successor ranks + Kasai (all positions
    indexed) or by unbounded comparison (filtered); both agree with the oracle-exact result and catch corruption."""
    text = tandem_text(3, 400_000)
    want = O.oracle_build(text, num_partitions=8, threads=4, **kw)
    r = device_build(S, text, 32, **kw)
    try:
        assert np.array_equal(r.sa_tensor().cpu().numpy().astype(np.uint32), want.sa)
        assert np.array_equal(r.lcp_tensor().cpu().numpy().astype(np.uint32), want.lcp)
        rep = r.verify()
        assert rep["ok"], rep
        assert rep["deferred_pairs"] > 0
        assert rep["method"] == (1 if kw.get("is_dna") and not kw.get("allow_ambiguity") else 2)
        assert rep["pairs_checked"] == r.num_suffixes - 1
        # corrupt one deep LCP value and one deep pair
        lcp, sa = r.lcp_tensor(), r.sa_tensor()
        deep = int(lcp.to(dtype=__import__("torch").int64).argmax().item())
        lcp[deep] -= 1
        bad = r.verify()
        assert bad["lcp_errors"] == 1 and bad["first_bad_rank"] == deep, bad
        lcp[deep] += 1
        a, b = sa[deep - 1].item(), sa[deep].item()
        sa[deep - 1], sa[deep] = b, a
        bad = r.verify()
        assert bad["order_errors"] >= 1, bad
    finally:
        r.free()


def test_verifier_sharded(S):
    """Every shard verifies itself (with the seam pair); the counts add up to the indexed positions."""
    text = rand_dna(9, 300_000, repeat_p=0.005, alphabet=b"ACGTN")
    world = 4
    import torch
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    shards = [S.build(S.SufrBuilderArgs(text=b"", is_dna=True), index_bits=64, result_memory=S.MEM_DEVICE,
                      device_text=(t.data_ptr(), t.numel()), rank=rk, world_size=world) for rk in range(world)]
    try:
        total, prev = 0, None
        for r in shards:
            if prev is not None and r.num_suffixes:
                r.patch_seam(prev)
            rep = r.verify(prev if r.num_suffixes else None)
            assert rep["order_errors"] + rep["lcp_errors"] + rep["duplicates"] + rep["not_indexed"] == 0, rep
            total += r.num_suffixes
            if r.num_suffixes:
                prev = r.last_suffix
        assert total == rep["expected_suffixes"]
    finally:
        for r in shards:
            r.free()


# ------------------------------------------------------------------ large comparisons with the oracle
@pytest.mark.parametrize("bits", [32, 64])
def test_oracle_200mbp_fast_path(S, bits):
    """BASELINE config 2 (iid ACGT, 24 records) at 200 Mbp: every SA and LCP entry against the oracle port."""
    w = workloads.config2_random(200_000_000)
    want = O.oracle_build(w.text, num_partitions=64, threads=16, index_bits=bits, is_dna=True)
    r = device_build(S, w.text, bits, is_dna=True)
    try:
        assert r.num_suffixes == want.num_suffixes
        assert np.array_equal(r.sa_tensor().cpu().numpy().astype(want.sa.dtype), want.sa)
        assert np.array_equal(r.lcp_tensor().cpu().numpy().astype(want.lcp.dtype), want.lcp)
        assert r.verify()["ok"]
    finally:
        r.free()


@pytest.mark.parametrize("name", ["config3", "config4"])
def test_oracle_100m_other_configs(S, name):
    """BASELINE configs 3 (protein, --max-query-len 32) and 4 (seed mask) at 100 M symbols: every SA and LCP entry
    against the oracle port, and the on-device verifier agrees."""
    w = workloads.ALL[name](100_000_000)
    want = O.oracle_build(w.text, num_partitions=64, threads=16, **w.flags)
    r = device_build(S, w.text, 32, **w.flags)
    try:
        assert r.num_suffixes == want.num_suffixes
        assert np.array_equal(r.sa_tensor().cpu().numpy().astype(np.uint32), want.sa)
        assert np.array_equal(r.lcp_tensor().cpu().numpy().astype(np.uint32), want.lcp)
        rep = r.verify()
        assert rep["ok"], rep
    finally:
        r.free()


def test_config5_100m_fully_verified(S):
    """BASELINE config 5 (tandem repeats, N runs, soft-mask) at 100 M symbols.  The reference's algorithm is quadratic
    on tandem arrays (the oracle port needs 77 s for 1 Mbp of this text, 326 s for 4 Mbp), so at this size the check is
    the full on-device verification -- itself pinned against the oracle on deep-repeat texts above -- and the oracle
    comparison of this generator runs at 300 kbp in test_gpu_parity.py."""
    w = workloads.config5(100_000_000)
    r = device_build(S, w.text, 32, **w.flags)
    try:
        rep = r.verify()
        assert rep["ok"], rep
        assert rep["pairs_checked"] == r.num_suffixes - 1 and rep["method"] == 2 and rep["max_lcp"] > 100_000
    finally:
        r.free()


# ------------------------------------------------------------------ one call, several GPUs (sufr_b200_create_multi)
def _ngpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("kw,bits", [(dict(is_dna=True), 64), (dict(is_dna=True, allow_ambiguity=True), 32),
                                     (dict(is_dna=True, seed_mask="1101101101"), 32), (dict(), 32)],
                         ids=["dna_u64", "dna_amb", "mask", "protein"])
def test_create_multi_file_is_byte_identical(S, tmp_path, kw, bits):
    """sufr_b200_create_multi over every visible GPU (a single-GPU box degenerates to one shard): the file is
    byte-identical to the oracle's."""
    ndev = max(1, min(8, _ngpus()))
    alphabet = b"ACGTN%" if kw.get("is_dna") else b"ACDEFGHIKLMNPQRSTVWY%"
    text = rand_dna(77, 400_000, repeat_p=0.01, alphabet=alphabet)
    starts, names = [0, 1000], ["chrA", "chrB"]
    want = O.oracle_build(text, num_partitions=16, threads=4, index_bits=bits, sequence_starts=starts,
                          sequence_names=names, **kw)
    out = tmp_path / "multi.sufr"
    info = S.create_multi(S.SufrBuilderArgs(text=text, path=str(out), sequence_starts=starts, sequence_names=names, **kw),
                          list(range(ndev)), index_bits=bits)
    assert info["num_suffixes"] == want.num_suffixes and info["text"] == want.text
    assert out.read_bytes() == want.file_bytes


def test_cli_devices_flag(S, tmp_path):
    import subprocess
    from conftest import GOLDEN, ROOT
    ndev = max(1, min(8, _ngpus()))
    out = tmp_path / "cli.sufr"
    devs = "0" if ndev == 1 else f"0-{ndev - 1}"
    p = subprocess.run([str(ROOT / "sufr_b200" / "sufr-b200"), "create", "--dna", "--devices", devs, "--log", "info",
                        "-o", str(out), str(GOLDEN / "inputs" / "long_dna_sequence.fa")], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    assert out.read_bytes() == (GOLDEN / "expected" / "long_dna_sequence.sufr").read_bytes()
    assert f"on {ndev} GPU" in p.stdout


# ------------------------------------------------------------------ 64-bit text positions (suffix_array.rs:460-470)
POS64_CASES = {
    "dna": (dict(is_dna=True), b"ACGTNacgtn%", 32),
    "dna_u64": (dict(is_dna=True), b"ACGT", 64),
    "dna_amb_soft": (dict(is_dna=True, allow_ambiguity=True, ignore_softmask=True), b"ACGTNacgtn%", 64),
    "protein": (dict(), b"ACDEFGHIKLMNPQRSTVWY%", 64),
    "mask": (dict(is_dna=True, seed_mask="1101101101"), b"ACGT", 32),
    "mql": (dict(max_query_len=300), b"ACGT", 64),
}


@pytest.mark.parametrize("case", list(POS64_CASES))
@pytest.mark.parametrize("world", [1, 3])
def test_64bit_positions_forced_on_short_texts(S, monkeypatch, case, world):
    """Texts of u32::MAX bytes and more take the 64-bit-position build (SufrBuilder::<u64>).  SUFR_B200_DEBUG_POS64
    forces that build on short texts, where the oracle can check it entry by entry, sharded and unsharded.  (The whole
    GPU suite also passes with the variable set: profiles/r2_gpu_suite_pos64.txt.)"""
    from sufr_b200.distributed import previous_last_suffix, shard_layout
    monkeypatch.setenv("SUFR_B200_DEBUG_POS64", "1")
    kw, alphabet, bits = POS64_CASES[case]
    text = rand_dna(seed_of(case), 120_000, repeat_p=0.02, alphabet=alphabet)
    want = O.oracle_build(text, num_partitions=8, threads=4, index_bits=bits, **kw)
    shards = [S.build(S.SufrBuilderArgs(text=text, **kw), index_bits=bits, rank=r, world_size=world) for r in range(world)]
    try:
        assert all(int(s.c.position_bits) == 64 for s in shards)
        meta = [(s.num_suffixes, s.first_suffix, s.last_suffix) for s in shards]
        offs, total = shard_layout(meta)
        for r, s in enumerate(shards):
            s.set_shard_layout(offs[r], total)
            prev = previous_last_suffix(meta, r)
            if prev is not None and s.num_suffixes:
                s.patch_seam(prev)
        assert total == want.num_suffixes
        assert np.array_equal(np.concatenate([s.sa for s in shards]), want.sa)
        assert np.array_equal(np.concatenate([s.lcp for s in shards]), want.lcp)
    finally:
        for s in shards:
            s.free()


def test_64bit_positions_deep_repeats_and_verifier(S, monkeypatch):
    monkeypatch.setenv("SUFR_B200_DEBUG_POS64", "1")
    text = tandem_text(11, 200_000)
    kw = dict(is_dna=True, allow_ambiguity=True)
    want = O.oracle_build(text, num_partitions=8, threads=4, index_bits=64, **kw)
    r = device_build(S, text, 64, **kw)
    try:
        assert int(r.c.position_bits) == 64 and int(r.c.doubling_rounds) > 0
        assert np.array_equal(r.sa_tensor().cpu().numpy().astype(np.uint64), want.sa)
        assert np.array_equal(r.lcp_tensor().cpu().numpy().astype(np.uint64), want.lcp)
        assert r.verify()["ok"]
    finally:
        r.free()


def test_long_text_needs_shards_and_u64(S):
    """Argument checks of the 64-bit branch: index_bits 32 is impossible, and one rank cannot hold >= 2^32 suffixes."""
    import ctypes as C
    from sufr_b200 import _lib
    ctx = S.default_context(0)
    args = S.builder._CArgs(S.SufrBuilderArgs(text=b""), text_ptr=0x1000, text_len=(1 << 32) + 5)
    res = _lib.Result()
    rc = _lib.lib().sufr_b200_build(ctx.handle, C.byref(args.c), 32, S.MEM_DEVICE, S.MEM_DEVICE, C.byref(res))
    assert rc == _lib.ERR_ARGUMENT and b"index_bits 64" in _lib.lib().sufr_b200_last_error()
    rc = _lib.lib().sufr_b200_build(ctx.handle, C.byref(args.c), 0, S.MEM_DEVICE, S.MEM_DEVICE, C.byref(res))
    assert rc == _lib.ERR_UNSUPPORTED and b"key-range shards" in _lib.lib().sufr_b200_last_error()
