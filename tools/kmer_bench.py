#!/usr/bin/env python
"""k-mer counting on a `.sufr` file on the GPU, measured (sufr_b200_index_kmer_spectrum, sufr_b200_index_kmers in
windows, sufr_b200_index_kmer_multiplicity in windows).

    python tools/kmer_bench.py [--bases 1000000000] [--index-bits 32] [--ks 21,31] [--window 16777216]
                               [--mult-window 268435456] [--out profiles/kmer_bench_1000Mbp_u32.json]

1. Writes the synthetic genome of bench.py (bench.record_layout + sufr_b200_synth_dna) with `create` to a file on a
   RAM disk (/dev/shm when present) and opens it into a device index (SufrIndex.open), as tools/mems_bench.py does.
2. For each k, best of --reps after a warm-up, host clock around calls that end in a device synchronise:
   - spectrum, cold: the call after one with another k, so it includes the text pass that makes the occurrence bitmap;
     and warm: the same k again (bitmap kept with the index);
   - enumeration of the k-mers with count >= 2 in windows of --window k-mers with their bytes (k-mers/s), and the
     same enumeration as one window (max_kmers = s), to compare the sum of the window times with one pass;
   - multiplicity of every position in windows of --mult-window positions (positions/s).
   Kernel time of each call from torch.profiler in a separate pass, and the bytes each pass must move over it, against
   7.7 TB/s.
3. Baseline: numpy on the host arrays of the same file (np.memmap of text, SA, LCP): the spectrum of the first k.
4. Checks: histogram sum = distinct, sum((i+1) h[i]) = occurrences (num_bins above the maximum count), the number of
   enumerated k-mers (count >= 2) + the count-1 bin = distinct, sum of multiplicities = sum of count^2, and the numpy
   spectrum equal to the GPU's.
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

HBM_BYTES_PER_S = 7.7e12
U64_MAX = 0xFFFFFFFFFFFFFFFF


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


def kernel_ms(fn):
    """Device time of all kernels of one call of fn under torch.profiler (ms)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = 0.0
    for ev in prof.key_averages():
        if "memcpy" in ev.key.lower() or "memset" in ev.key.lower():
            continue
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        total += (t or 0) / 1000.0
    return total


def best(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return min(times)


def numpy_spectrum(text, sa, lcp, starts, k, num_bins):
    """The spectrum of a DNA index from its host arrays: occurrences from the text, groups from LCP < k."""
    n = len(text)
    ex = ~np.isin(text, np.frombuffer(b"ACGT", np.uint8))
    ex[-1] = True
    st = np.asarray(starts, np.int64)
    ex[st[st > 0] - 1] = True
    pos = np.flatnonzero(ex)
    nxt = pos[np.searchsorted(pos, np.arange(n))]
    occ = (nxt - np.arange(n)) >= k
    heads = np.flatnonzero(lcp < k)
    if len(heads) == 0 or heads[0] != 0:
        heads = np.concatenate([[0], heads])
    counts = np.add.reduceat(occ[sa].astype(np.int64), heads)
    counts = counts[counts > 0]
    h = np.bincount(np.minimum(counts, num_bins) - 1, minlength=num_bins).astype(np.uint64)
    return h, len(counts), int(counts.sum()), int(counts.max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=1_000_000_000)
    ap.add_argument("--index-bits", type=int, default=32, choices=[32, 64])
    ap.add_argument("--ks", default="21,31")
    ap.add_argument("--num-bins", type=int, default=10000)
    ap.add_argument("--window", type=int, default=1 << 24)
    ap.add_argument("--mult-window", type=int, default=1 << 28)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-baseline", action="store_true")
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out", default=None, help="default: profiles/kmer_bench_<Mbp>Mbp_u<bits>.json")
    a = ap.parse_args()
    out_path = a.out or str(ROOT / "profiles" / f"kmer_bench_{a.bases // 1_000_000}Mbp_u{a.index_bits}.json")
    ks = [int(x) for x in a.ks.split(",")]
    gpu = gpu_identity()
    text_len, starts = bench.record_layout(a.bases)
    names = [f"chr{i + 1}" for i in range(len(starts))]
    st = np.asarray(starts, dtype=np.uint64)
    ctx = S.Context(0)
    d_text = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    check(_lib.lib().sufr_b200_synth_dna(ctx.handle, d_text.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                         ord("%")))
    tmpdir = tempfile.mkdtemp(prefix="sufr_kmers_", dir=a.dir)
    path = os.path.join(tmpdir, "genome.sufr")
    L = _lib.lib()
    result = {"workload": {"bases": a.bases, "text_len": text_len, "records": len(starts), "index_bits": a.index_bits,
                           "file_dir": a.dir, "ks": ks, "window": a.window, "mult_window": a.mult_window,
                           "reps": a.reps},
              "gpu": gpu, "k": {}}
    try:
        cargs = S.SufrBuilderArgs(text=d_text.cpu().numpy().tobytes(), path=path, is_dna=True, sequence_starts=starts,
                                  sequence_names=names)
        S.create_multi(cargs, [0], index_bits=a.index_bits)
        del cargs, d_text
        torch.cuda.empty_cache()
        idx = S.SufrIndex.open(path, ctx=ctx)
        n, s, w = idx._n, idx._s, a.index_bits // 8
        result["workload"]["suffixes"] = s
        hist = np.zeros(a.num_bins, np.uint64)
        d, o, m = C.c_uint64(), C.c_uint64(), C.c_uint64()
        per = a.window
        cols = [np.zeros(max(per, 1), np.uint64) for _ in range(3)]
        num, nxt = C.c_uint64(), C.c_uint64()
        mult = np.zeros(min(a.mult_window, n), np.uint32)

        def spectrum(k):
            check(L.sufr_b200_index_kmer_spectrum(idx._h, k, a.num_bins, hist.ctypes.data, C.byref(d), C.byref(o),
                                                  C.byref(m)))

        def enumerate_windows(k, max_kmers, buf):
            first, got, win_times = 0, 0, []
            while first < s:
                t0 = time.perf_counter()
                check(L.sufr_b200_index_kmers(idx._h, k, 2, U64_MAX, first, max_kmers, C.byref(num), C.byref(nxt),
                                              *[c.ctypes.data for c in cols], None if buf is None else buf.ctypes.data))
                win_times.append(time.perf_counter() - t0)
                got += int(num.value)
                first = int(nxt.value)
            return got, win_times

        def multiplicity(k, on_window=None):
            for f in range(0, n, a.mult_window):
                ln = min(a.mult_window, n - f)
                check(L.sufr_b200_index_kmer_multiplicity(idx._h, k, f, ln, mult.ctypes.data))
                if on_window:
                    on_window(mult[:ln])

        for k in ks:
            other = ks[0] + ks[-1] - k if len(ks) > 1 else k + 1
            r = {}
            # ---- spectrum, cold (after another k: includes the text pass) and warm
            cold = []
            for _ in range(a.reps):
                spectrum(other)
                t0 = time.perf_counter()
                spectrum(k)
                cold.append(time.perf_counter() - t0)
            warm = best(lambda: spectrum(k), a.reps)
            h = hist.copy()
            distinct, occurrences, max_count = d.value, o.value, m.value
            spectrum(other)
            cold_kernel = kernel_ms(lambda: spectrum(k))
            warm_kernel = kernel_ms(lambda: spectrum(k))
            r["spectrum"] = {"cold_s": min(cold), "warm_s": warm, "cold_kernel_ms": cold_kernel,
                             "warm_kernel_ms": warm_kernel, "distinct": distinct, "occurrences": occurrences,
                             "max_count": max_count, "histogram_head": h[:10].tolist(),
                             "last_bin": int(h[-1])}
            # bytes a pass must move: the text pass reads the text once and writes / reads the n-bit bitmaps;
            # the rank pass reads SA and LCP twice (reduce + apply of the scan) and gathers one 32-byte sector of the
            # occurrence bitmap per rank and read
            text_bytes = n + 4 * (n // 8)
            rank_bytes = 2 * (2 * w * s) + 2 * 32 * s
            min_bytes = n + 2 * w * s
            r["spectrum"]["bytes_cold"] = text_bytes + rank_bytes
            r["spectrum"]["bytes_warm"] = rank_bytes
            r["spectrum"]["min_bytes"] = min_bytes
            r["spectrum"]["hbm_share_warm_kernel"] = rank_bytes / (warm_kernel / 1e3) / HBM_BYTES_PER_S
            r["spectrum"]["roofline_ms_min_bytes"] = min_bytes / HBM_BYTES_PER_S * 1e3

            # ---- enumeration, count >= 2, in windows and as one window
            buf = np.zeros(per * k, np.uint8)
            listed, win = enumerate_windows(k, per, buf)
            wtimes = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                listed, win = enumerate_windows(k, per, buf)
                wtimes.append(time.perf_counter() - t0)
            r["kmers_ge2"] = {"listed": listed, "windows": len(win), "time_s": min(wtimes),
                              "kmers_per_s": listed / min(wtimes), "sum_window_s": sum(win)}
            one_cols = cols
            if listed <= 4 * per:  # one window: the whole enumeration in one call, without the bytes
                cols = [np.zeros(max(listed, 1), np.uint64) for _ in range(3)]
                t0 = time.perf_counter()
                got1, _ = enumerate_windows(k, s, None)
                r["kmers_ge2"]["one_window_s"] = time.perf_counter() - t0
                assert got1 == listed
                cols = one_cols
            r["kmers_ge2"]["kernel_ms"] = kernel_ms(lambda: enumerate_windows(k, per, buf))

            # ---- multiplicity in windows
            mtimes = []
            sq = [0]

            def acc(x):
                sq[0] += int(x.astype(np.int64).sum())
            multiplicity(k, acc)
            mult_sum = sq[0]
            for _ in range(a.reps):
                t0 = time.perf_counter()
                multiplicity(k)
                mtimes.append(time.perf_counter() - t0)
            mk = kernel_ms(lambda: multiplicity(k))
            windows = -(-n // a.mult_window)
            # the forward scan once per k (SA + LCP twice, a sector per rank twice, the u32 counts written), then per
            # window the reverse scan (LCP and the counts twice, SA and a sector once) and the output once
            mbytes = (2 * (2 * w * s) + 64 * s + 4 * s) + windows * (3 * w * s + 8 * s + 32 * s) + n * 4
            r["multiplicity"] = {"windows": windows, "time_s": min(mtimes), "positions_per_s": n / min(mtimes),
                                 "kernel_ms": mk, "bytes": mbytes,
                                 "hbm_share_kernel": mbytes / (mk / 1e3) / HBM_BYTES_PER_S}

            # ---- consistency
            top_ok = max_count < a.num_bins
            c = {"hist_sum_is_distinct": int(h.sum()) == distinct}
            if top_ok:
                c["weighted_sum_is_occurrences"] = int(sum((i + 1) * int(x) for i, x in enumerate(h.tolist()))) == occurrences
                c["listed_plus_ones_is_distinct"] = listed + int(h[0]) == distinct
                c["mult_sum_is_sum_count_sq"] = mult_sum == int(sum((i + 1) ** 2 * int(x) for i, x in
                                                                    enumerate(h.tolist())))
            r["checks"] = c
            result["k"][str(k)] = r

        if not a.no_baseline:
            k = ks[0]
            info = idx.info
            mm = np.memmap(path, dtype=np.uint8, mode="r")
            udt = np.uint32 if a.index_bits == 32 else np.uint64
            text = np.asarray(mm[info["text_pos"]:info["text_pos"] + n])
            sa = np.asarray(mm[info["sa_pos"]:info["sa_pos"] + s * w]).view(udt)
            lcp = np.asarray(mm[info["lcp_pos"]:info["lcp_pos"] + s * w]).view(udt)
            t0 = time.perf_counter()
            nh, nd, no, nm = numpy_spectrum(text, sa, lcp, starts, k, a.num_bins)
            tb = time.perf_counter() - t0
            spectrum(k)
            result["baseline_numpy"] = {"k": k, "spectrum_s": tb, "equal": bool(np.array_equal(nh, hist) and
                                                                                (nd, no, nm) == (d.value, o.value,
                                                                                                 m.value))}
            result["baseline_numpy"]["speedup_cold"] = tb / result["k"][str(k)]["spectrum"]["cold_s"]
        idx.close()
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    Path(out_path).parent.mkdir(parents=True, exist_ok=True)
    Path(out_path).write_text(line + "\n")


if __name__ == "__main__":
    main()
