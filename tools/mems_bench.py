#!/usr/bin/env python
"""Matching statistics and MEMs of reads against a `.sufr` file on the GPU, measured (sufr_b200_index_matching_stats,
sufr_b200_index_mems + windowed sufr_b200_index_hits).

    python tools/mems_bench.py [--bases 1000000000] [--reads 100000] [--random-reads 10000] [--min-len 20]
                               [--out profiles/mems_bench_1000Mbp_u32.json]

1. Writes the synthetic genome of bench.py (bench.record_layout + sufr_b200_synth_dna) with `create` to a file on a
   RAM disk (/dev/shm when present) and opens it into a device index (SufrIndex.open), as tools/file_query_bench.py does.
2. Reads: --reads of --read-len bases sampled from the text with --sub-rate substitutions, plus --random-reads uniform
   random reads, in one batch.
3. Times, best of --reps after a warm-up, with host buffers in and out and a host clock around calls that end in a
   device synchronise: matching statistics of every position (positions/s); MEMs of at least --min-len plus every
   hit window (MEMs/s, hits/s).  Kernel time of both from torch.profiler in a separate pass.
4. Baseline: the same matching statistics from Python, one SufrIndex.search call per substring (seeded with
   ms[i] >= ms[i-1] - 1, so about two calls per position), on the first --baseline-reads reads.
5. Checks, on --check-positions sampled positions: search(q[i, i+ms)) gives the same rank range, q[i, i+ms+1) occurs
   nowhere, and the range's first and last suffixes start with q[i, i+ms).  The MEM list equals the one derived from
   the matching statistics on the host, the hit offsets their counts, and sampled hits the suffix array entries.
Prints one JSON line with the GPU's name and power limit read in the same run, and writes it to --out."""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402
import bench  # noqa: E402
import sufr_b200 as S  # noqa: E402
from sufr_b200 import _lib  # noqa: E402

NONE = np.uint64(0xFFFFFFFFFFFFFFFF)


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    power = None
    try:  # read-only query
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:
        pass
    return {"name": name, "power_limit_w": power}


def check(rc):
    assert rc == 0, _lib.lib().sufr_b200_last_error().decode()


class Runner:
    """The two calls through the C ABI with preallocated host buffers."""

    def __init__(self, idx, blob, offs, window):
        self.idx, self.blob, self.offs, self.window = idx, blob, offs, window
        self.nq, self.total = len(offs) - 1, int(offs[-1])
        self.ms = [np.zeros(self.total, np.uint64) for _ in range(3)]
        self.mem = [np.zeros(self.total, np.uint64) for _ in range(5)]
        self.ho = np.zeros(self.total + 1, np.uint64)
        self.hit = [np.zeros(window, np.uint64) for _ in range(3)]
        self.num = C.c_uint64()

    def matching_stats(self):
        check(_lib.lib().sufr_b200_index_matching_stats(self.idx._h, self.blob.ctypes.data, self.offs.ctypes.data,
                                                        self.nq, *[a.ctypes.data for a in self.ms]))
        return self.ms

    def mems(self, min_len, on_window=None):
        check(_lib.lib().sufr_b200_index_mems(self.idx._h, self.blob.ctypes.data, self.offs.ctypes.data, self.nq,
                                              min_len, C.byref(self.num), *[a.ctypes.data for a in self.mem],
                                              self.ho.ctypes.data))
        k = int(self.num.value)
        total = int(self.ho[k])
        for first in range(0, total, self.window):
            n = min(self.window, total - first)
            check(_lib.lib().sufr_b200_index_hits(self.idx._h, first, n, *[a.ctypes.data for a in self.hit]))
            if on_window:
                on_window(first, n, [a[:n] for a in self.hit])
        return k, total


def host_mems(ms, offs, min_len):
    """Indices j of the batch bytes that start a MEM (include/sufr_b200.h), from the matching statistics."""
    start = np.zeros(len(ms), bool)
    o = offs[:-1][offs[:-1] < offs[1:]].astype(np.int64)
    start[o] = True
    prev = np.concatenate([[np.uint64(0)], ms[:-1]])
    return np.flatnonzero((ms >= min_len) & (start | (prev <= ms)))


def baseline(idx, reads):
    """Matching statistics from Python, one search call per substring."""
    out = []
    for q in reads:
        ms = []
        for i in range(len(q)):
            ln = max(ms[-1] - 1, 0) if ms else 0
            while i + ln < len(q) and idx.search([q[i:i + ln + 1]], None, True)[0] is not None:
                ln += 1
            ms.append(ln)
        out.append(ms)
    return out


def kernel_times(fn):
    """Device time per kernel name of one call of fn under torch.profiler (ms)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t:
            out[ev.key] = out.get(ev.key, 0.0) + t / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=1_000_000_000)
    ap.add_argument("--index-bits", type=int, default=32, choices=[32, 64])
    ap.add_argument("--reads", type=int, default=100_000)
    ap.add_argument("--random-reads", type=int, default=10_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--sub-rate", type=float, default=0.01)
    ap.add_argument("--min-len", type=int, default=20)
    ap.add_argument("--window", type=int, default=1 << 24)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-reads", type=int, default=20)
    ap.add_argument("--check-positions", type=int, default=20_000)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out", default=None, help="default: profiles/mems_bench_<Mbp>Mbp_u<bits>.json")
    a = ap.parse_args()
    out_path = a.out or str(ROOT / "profiles" / f"mems_bench_{a.bases // 1_000_000}Mbp_u{a.index_bits}.json")
    gpu = gpu_identity()
    text_len, starts = bench.record_layout(a.bases)
    names = [f"chr{i + 1}" for i in range(len(starts))]
    st = np.asarray(starts, dtype=np.uint64)
    ctx = S.Context(0)
    d_text = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    check(_lib.lib().sufr_b200_synth_dna(ctx.handle, d_text.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                         ord("%")))

    # reads: substrings with substitutions, then uniform random reads
    g = torch.Generator(device="cuda").manual_seed(13)
    L = a.read_len
    p = torch.randint(0, text_len - L - 1, (a.reads,), device="cuda", generator=g)
    sampled = d_text[p[:, None] + torch.arange(L, device="cuda")[None, :]]
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    sub = torch.rand(sampled.shape, device="cuda", generator=g) < a.sub_rate
    sampled = torch.where(sub, acgt[torch.randint(0, 4, sampled.shape, device="cuda", generator=g)], sampled)
    rand = acgt[torch.randint(0, 4, (a.random_reads, L), device="cuda", generator=g)]
    reads = torch.cat([sampled, rand]).cpu().numpy()
    blob = reads.reshape(-1).copy()
    offs = np.arange(len(reads) + 1, dtype=np.uint64) * L
    read_bytes = [reads[i].tobytes() for i in range(len(reads))]

    tmpdir = tempfile.mkdtemp(prefix="sufr_mems_", dir=a.dir)
    path = os.path.join(tmpdir, "genome.sufr")
    try:
        cargs = S.SufrBuilderArgs(text=d_text.cpu().numpy().tobytes(), path=path, is_dna=True, sequence_starts=starts,
                                  sequence_names=names)
        S.create_multi(cargs, [0], index_bits=a.index_bits)
        del cargs
        del d_text
        torch.cuda.empty_cache()
        idx = S.SufrIndex.open(path, ctx=ctx)
        run = Runner(idx, blob, offs, a.window)
        positions = run.total

        # ---- matching statistics
        run.matching_stats()  # warm-up
        times = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            run.matching_stats()
            times.append(time.perf_counter() - t0)
        ms_s = min(times)
        ms, rb, re_ = (x.copy() for x in run.ms)

        # ---- MEMs + every hit window
        run.mems(a.min_len)  # warm-up
        mtimes = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            num_mems, num_hits = run.mems(a.min_len)
            mtimes.append(time.perf_counter() - t0)
        mem_s = min(mtimes)

        # ---- kernel time (separate pass under the profiler)
        k_ms = kernel_times(run.matching_stats)
        k_mem = kernel_times(lambda: run.mems(a.min_len))
        ms_kernel = sum(v for k, v in k_ms.items() if "matching_stats_kernel" in k)

        # ---- checks
        rng = np.random.default_rng(5)
        sample = np.sort(rng.choice(positions, min(a.check_positions, positions), replace=False))
        subs, ranges, longer, bad_bytes = [], [], [], 0
        for j in sample.tolist():
            qi, i = j // L, j % L
            q, k = read_bytes[qi], int(ms[j])
            if k:
                subs.append(q[i:i + k])
                ranges.append((int(rb[j]), int(re_[j])))
                for r in (int(rb[j]), int(re_[j]) - 1):
                    suf = int(idx.suffixes(r, 1)[0])
                    bad_bytes += idx.string_at(suf, k) != q[i:i + k]
            elif rb[j] != NONE or re_[j] != NONE:
                bad_bytes += 1
            if i + k < L:
                longer.append(q[i:i + k + 1])
        range_ok = idx.search(subs, None, True) == ranges
        longer_ok = all(x is None for x in idx.search(longer, None, True))
        want_j = host_mems(ms, offs, a.min_len)
        run.mems(a.min_len)
        k = int(run.num.value)
        mq, mp, ml, mb, me = (x[:k] for x in run.mem)
        mems_ok = bool(k == len(want_j) and np.array_equal(mq * np.uint64(L) + mp, want_j.astype(np.uint64)) and
                       np.array_equal(ml, ms[want_j]) and np.array_equal(mb, rb[want_j]) and
                       np.array_equal(me, re_[want_j]))
        counts = (me - mb).astype(np.int64)
        offsets_ok = run.ho[:k + 1].tolist() == [0] + np.cumsum(counts).tolist()
        # sampled hits: the first hit of every 97th MEM is SA[rank_begin]
        hit_bad, hit_checked = 0, 0
        for m in range(0, k, 97):
            h = int(run.ho[m])
            check(_lib.lib().sufr_b200_index_hits(idx._h, h, 1, *[x.ctypes.data for x in run.hit]))
            hit_bad += int(run.hit[0][0]) != int(idx.suffixes(int(mb[m]), 1)[0])
            hit_checked += 1

        # ---- baseline on a subset
        sub_reads = read_bytes[:a.baseline_reads]
        t0 = time.perf_counter()
        base = baseline(idx, sub_reads)
        base_s = time.perf_counter() - t0
        base_pos = sum(len(q) for q in sub_reads)
        base_same = all(np.array_equal(np.asarray(b_, np.uint64), ms[i * L:(i + 1) * L]) for i, b_ in enumerate(base))
        info = idx.info
        idx.close()
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    ok = bool(range_ok and longer_ok and bad_bytes == 0 and mems_ok and offsets_ok and hit_bad == 0 and base_same)
    res = {"metric": "matching statistics positions/s; MEMs + all their hits, MEMs/s and hits/s",
           "gpu": gpu, "bases": a.bases, "text_len": text_len, "index_bits": a.index_bits,
           "num_suffixes": info["num_suffixes"], "records": len(starts),
           "reads": {"sampled": a.reads, "random": a.random_reads, "len": L, "sub_rate": a.sub_rate},
           "positions": positions,
           "matching_stats": {"s": ms_s, "all_s": times, "positions_per_s": positions / ms_s,
                              "kernel_ms": ms_kernel, "kernel_positions_per_s": positions / (ms_kernel / 1000.0)
                              if ms_kernel else None,
                              "positions_with_match": int((ms > 0).sum()), "mean_ms": float(ms.mean())},
           "mems": {"min_len": a.min_len, "mems": num_mems, "hits": num_hits, "s": mem_s, "all_s": mtimes,
                    "mems_per_s": num_mems / mem_s, "hits_per_s": num_hits / mem_s},
           "profiler_ms": {"matching_stats_call": k_ms, "mems_call": k_mem},
           "baseline": {"reads": len(sub_reads), "positions": base_pos, "s": base_s,
                        "positions_per_s": base_pos / base_s, "same_ms": base_same,
                        "speedup": (positions / ms_s) / (base_pos / base_s),
                        "note": "Python loop, one SufrIndex.search per substring, seeded with ms[i-1] - 1"},
           "check": {"ok": ok, "positions_checked": len(sample), "ranges_equal_search": range_ok,
                     "one_byte_longer_absent": longer_ok, "range_end_bytes_bad": bad_bytes,
                     "mems_equal_host_derivation": mems_ok, "hit_offsets_ok": offsets_ok,
                     "hits_checked": hit_checked, "hits_bad": hit_bad},
           "reps": a.reps,
           "note": "timed region: queries uploaded from host memory and every output downloaded to host memory, host "
                   "clock around calls that end in a device synchronise, best of reps after a warm-up; the index was "
                   "opened from a file on a RAM disk; kernel times from torch.profiler in a separate pass"}
    line = json.dumps(res)
    print(line)
    Path(out_path).parent.mkdir(parents=True, exist_ok=True)
    Path(out_path).write_text(line + "\n")
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
