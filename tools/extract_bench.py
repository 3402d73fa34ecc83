#!/usr/bin/env python
"""extract and list on a `.sufr` FILE opened into a device index, measured (sufr_b200_index_extract / _list; mirrors
SufrFile::extract / SufrFile::list).

    python tools/extract_bench.py [--bases 1000000000] [--reps 3]

1. Writes the synthetic genome of tools/file_query_bench.py (bench.record_layout + sufr_b200_synth_dna, u32) with
   `create` to a RAM disk (/dev/shm when present) and opens it with SufrIndex.open.
2. Workloads, each end to end through the C ABI with host buffers (locate + every extract window, or every list
   window), best of --reps:
     long   4 M 24-mers sampled from the text, prefix_len = suffix_len = 50
     short  10 k 8-mers (about 150 M hits), prefix_len = suffix_len = 10
     whole  64 hits with suffix_len unset: every region runs to the end of its record (tens of MB each)
     list   10 M rows from a random rank, len = 32
3. One more pass per workload under torch.profiler: the device time of gather_regions_kernel (reported against
   HBM bandwidth, 2 bytes of traffic per output byte) and of the device-to-host copies.
4. Checks the first window and a middle window of every workload against a numpy restatement over the file's text,
   suffix array and LCP sections (memory-mapped), with the hits from sufr_b200_index_hits.
5. The old way on a subset: device locate + hits, then one numpy slice of the memory-mapped text per hit.
Prints one JSON line with the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import shutil
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import torch  # noqa: E402
import bench  # noqa: E402
import file_query_bench as fqb  # noqa: E402
import sufr_b200 as S  # noqa: E402
from sufr_b200 import _lib  # noqa: E402

U64_MAX = 0xFFFFFFFFFFFFFFFF
HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


class Extractor:
    """locate, then every extract window, through the C ABI with preallocated host buffers."""

    def __init__(self, idx, window, max_bytes):
        self.idx, self.window, self.max_bytes = idx, window, max_bytes
        self.cols = [np.zeros(window, np.uint64) for _ in range(4)]
        self.offs = np.zeros(window + 1, np.uint64)
        self.buf = np.zeros(max_bytes, np.uint8)
        self.locator = fqb.Runner(idx, 1)

    def extract(self, first, count, P, S_):
        num = C.c_uint64()
        rc = _lib.lib().sufr_b200_index_extract(self.idx._h, first, count, P, S_, self.max_bytes, C.byref(num),
                                                *[c.ctypes.data for c in self.cols], self.offs.ctypes.data,
                                                self.buf.ctypes.data)
        assert rc == 0, _lib.lib().sufr_b200_last_error()
        k = int(num.value)
        assert k > 0, "a region larger than the buffer"
        return k

    def run(self, blob, offs, P, S_):
        _, _, ho = self.locator.locate(blob, offs)
        total, first, nbytes = int(ho[-1]), 0, 0
        while first < total:
            k = self.extract(first, min(self.window, total - first), P, S_)
            nbytes += int(self.offs[k])
            first += k
        return total, nbytes


class Lister(Extractor):
    def list(self, first, count, L):
        num = C.c_uint64()
        rc = _lib.lib().sufr_b200_index_list(self.idx._h, first, count, L, self.max_bytes, C.byref(num),
                                             self.cols[0].ctypes.data, self.cols[1].ctypes.data, self.offs.ctypes.data,
                                             self.buf.ctypes.data)
        assert rc == 0, _lib.lib().sufr_b200_last_error()
        return int(num.value)

    def run(self, first_rank, rows, L):
        r, end, nbytes = first_rank, first_rank + rows, 0
        while r < end:
            k = self.list(r, min(self.window, end - r), L)
            nbytes += int(self.offs[k])
            r += k
        return rows, nbytes


def restate_regions(text, st, suf, P, S_):
    """region (start, end) relative to the record, and its absolute source, of hits at suffixes suf"""
    n = len(text)
    seq = np.searchsorted(st, suf, side="right").astype(np.int64) - 1
    a = np.where(seq < 0, 0, st[np.maximum(seq, 0)]).astype(np.uint64)
    nxt = np.append(st[1:], np.uint64(n))
    e = np.where(seq < 0, st[0] if len(st) else n, nxt[np.maximum(seq, 0)]).astype(np.uint64)
    rel = suf - a
    start = rel - np.minimum(rel, np.uint64(P))
    end = e - a if S_ == U64_MAX else np.minimum(rel + np.uint64(S_), e - a)
    return np.where(seq < 0, U64_MAX, seq).astype(np.uint64), start, end, a


def profile_pass(fn):
    """(gather kernel ms, gather launches, device-to-host copy ms) of one call of fn under torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    k_us, k_n, c_us = 0.0, 0, 0.0
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        t = getattr(ev, "cuda_time_total", 0.0) if t is None else t
        if "gather_regions_kernel" in ev.key:
            k_us += t
            k_n += ev.count
        elif "DtoH" in ev.key:
            c_us += t
    return k_us / 1e3, k_n, c_us / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=1_000_000_000)
    ap.add_argument("--long-queries", type=int, default=4_000_000)
    ap.add_argument("--short-queries", type=int, default=10_000)
    ap.add_argument("--whole-hits", type=int, default=64)
    ap.add_argument("--list-rows", type=int, default=10_000_000)
    ap.add_argument("--window", type=int, default=1 << 24)
    ap.add_argument("--max-bytes", type=int, default=1 << 31)
    ap.add_argument("--check-hits", type=int, default=1 << 17)
    ap.add_argument("--old-hits", type=int, default=200_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    a = ap.parse_args()
    gpu = fqb.gpu_identity()
    text_len, starts = bench.record_layout(a.bases)
    names = [f"chr{i + 1}" for i in range(len(starts))]
    st = np.asarray(starts, dtype=np.uint64)
    ctx = S.Context(0)
    d_text = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    assert _lib.lib().sufr_b200_synth_dna(ctx.handle, d_text.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                          ord("%")) == 0
    g = torch.Generator(device="cuda").manual_seed(12)

    def substrings(n, L):
        p = torch.randint(0, text_len - L - 1, (n,), device="cuda", generator=g)
        return d_text[p[:, None] + torch.arange(L, device="cuda")[None, :]].contiguous()

    workloads = {
        "long": (fqb.blob_of(substrings(a.long_queries, 24)), 50, 50),
        "short": (fqb.blob_of(substrings(a.short_queries, 8)), 10, 10),
        "whole": (fqb.blob_of(substrings(a.whole_hits, 24)), 0, U64_MAX),
    }
    tmpdir = tempfile.mkdtemp(prefix="sufr_extract_", dir=a.dir)
    path = os.path.join(tmpdir, "genome.sufr")
    try:
        cargs = S.SufrBuilderArgs(text=d_text.cpu().numpy().tobytes(), path=path, is_dna=True, sequence_starts=starts,
                                  sequence_names=names)
        S.create_multi(cargs, [0], index_bits=32)
        del cargs, d_text
        torch.cuda.empty_cache()
        ctx.trim()
        info = S.file_info(path)
        mm = np.memmap(path, dtype=np.uint8, mode="r")
        text = mm[info["text_pos"]:info["text_pos"] + info["text_len"]]
        sa = mm[info["sa_pos"]:info["lcp_pos"]].view(np.uint32)
        lcp = mm[info["lcp_pos"]:info["lcp_pos"] + 4 * info["num_suffixes"]].view(np.uint32)
        idx = S.SufrIndex.open(path, ctx=ctx)
        ex = Extractor(idx, a.window, a.max_bytes)
        results, ok = {}, True
        for key, ((blob, offs), P, S_) in workloads.items():
            total, nbytes = ex.run(blob, offs, P, S_)  # warm-up
            times = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                ex.run(blob, offs, P, S_)
                times.append(time.perf_counter() - t0)
            dt = min(times)
            k_ms, k_n, c_ms = profile_pass(lambda: ex.run(blob, offs, P, S_))
            c_bytes = nbytes + 40 * total + 24 * (len(offs) - 1)  # bytes, 4 columns + offsets, locate's outputs
            # checks: the first window and a middle window
            checked, bad = 0, 0
            for first in sorted({0, total // 2}):
                cnt = min(a.check_hits, total - first)
                if cnt <= 0:
                    continue
                suf, _, _ = idx.hits(first, cnt)
                k = ex.extract(first, cnt, P, S_)
                seq, start, end, rec = restate_regions(text, st, suf[:k], P, S_)
                got = [c[:k] for c in ex.cols]
                bad += int((got[0] != suf[:k]).sum() + (got[1] != seq).sum() + (got[2] != start).sum() +
                           (got[3] != end).sum())
                o = ex.offs[:k + 1]
                bad += int((np.diff(o) != end - start).sum())
                src = rec + start
                for i in range(0, k, max(1, k // 4096)):  # every region up to 4096 of them, byte for byte
                    if ex.buf[int(o[i]):int(o[i + 1])].tobytes() != text[int(src[i]):int(src[i] + end[i] - start[i])].tobytes():
                        bad += 1
                checked += k
            # the old way on a subset: device locate + hits, one numpy slice of the mapped text per hit
            old_n = min(a.old_hits, total)
            t0 = time.perf_counter()
            _, _, ho = ex.locator.locate(blob, offs)
            suf, seqs, _ = idx.hits(0, old_n)
            nxt = np.append(st[1:], np.uint64(len(text))).tolist()
            stl = st.tolist()
            old_bytes = 0
            for p, s_ in zip(suf.tolist(), seqs.tolist()):
                a0, e0 = stl[s_], nxt[s_]
                rel = p - a0
                b0 = a0 + rel - min(rel, P)
                e1 = e0 if S_ == U64_MAX else min(a0 + rel + S_, e0)
                old_bytes += len(bytes(text[b0:e1]))
            old_s = time.perf_counter() - t0
            results[key] = {"queries": len(offs) - 1, "query_len": int(offs[1]), "prefix_len": P,
                            "suffix_len": None if S_ == U64_MAX else S_, "hits": total, "bytes": nbytes,
                            "s": dt, "all_s": times, "hits_per_s": total / dt, "bytes_per_s": nbytes / dt,
                            "gather_kernel_ms": k_ms, "gather_launches": k_n,
                            "gather_hbm_bytes_per_s": 2 * nbytes / (k_ms / 1e3) if k_ms else None,
                            "gather_share_of_hbm": (2 * nbytes / (k_ms / 1e3)) / HBM_BYTES_PER_S if k_ms else None,
                            "d2h_ms": c_ms, "d2h_bytes": c_bytes, "d2h_gb_per_s": c_bytes / (c_ms / 1e3) / 1e9 if c_ms else None,
                            "gather_over_d2h": k_ms / c_ms if c_ms else None,
                            "checked": checked, "bad": bad,
                            "old_path": {"hits": old_n, "bytes": old_bytes, "s": old_s},
                            "speedup_vs_old_path": (total / dt) / (old_n / old_s) if old_s else None}
            ok = ok and bad == 0
        # list
        lister = Lister(idx, a.window, a.max_bytes)
        rows = min(a.list_rows, info["num_suffixes"])
        first_rank = int(np.random.default_rng(5).integers(0, info["num_suffixes"] - rows + 1))
        _, nbytes = lister.run(first_rank, rows, 32)
        times = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            lister.run(first_rank, rows, 32)
            times.append(time.perf_counter() - t0)
        dt = min(times)
        k_ms, k_n, c_ms = profile_pass(lambda: lister.run(first_rank, rows, 32))
        c_bytes = nbytes + 24 * rows  # bytes, suffix, lcp, offsets
        checked, bad = 0, 0
        for r0 in sorted({first_rank, first_rank + rows // 2}):
            cnt = min(a.check_hits, first_rank + rows - r0)
            k = lister.list(r0, cnt, 32)
            want_suf = sa[r0:r0 + k].astype(np.uint64)
            bad += int((lister.cols[0][:k] != want_suf).sum() + (lister.cols[1][:k] != lcp[r0:r0 + k]).sum())
            ln = np.minimum(np.uint64(32), np.uint64(len(text)) - want_suf)
            o = lister.offs[:k + 1]
            bad += int((np.diff(o) != ln).sum())
            for i in range(0, k, max(1, k // 4096)):
                p = int(want_suf[i])
                if lister.buf[int(o[i]):int(o[i + 1])].tobytes() != text[p:p + int(ln[i])].tobytes():
                    bad += 1
            checked += k
        results["list"] = {"rows": rows, "first_rank": first_rank, "len": 32, "bytes": nbytes, "s": dt, "all_s": times,
                           "rows_per_s": rows / dt, "bytes_per_s": nbytes / dt, "gather_kernel_ms": k_ms,
                           "gather_launches": k_n,
                           "gather_hbm_bytes_per_s": 2 * nbytes / (k_ms / 1e3) if k_ms else None,
                           "gather_share_of_hbm": (2 * nbytes / (k_ms / 1e3)) / HBM_BYTES_PER_S if k_ms else None,
                           "d2h_ms": c_ms, "d2h_bytes": c_bytes,
                           "d2h_gb_per_s": c_bytes / (c_ms / 1e3) / 1e9 if c_ms else None,
                           "gather_over_d2h": k_ms / c_ms if c_ms else None, "checked": checked, "bad": bad}
        ok = ok and bad == 0
        idx.close()
        del mm, text, sa, lcp
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    out = {"metric": "extract hits/s and bytes/s, list rows/s and bytes/s (device index opened from a .sufr file)",
           "gpu": gpu, "bases": a.bases, "text_len": text_len, "index_bits": 32, "records": len(starts),
           "workloads": results, "window": a.window, "max_bytes": a.max_bytes, "reps": a.reps,
           "note": "s: host clock, best of reps, queries uploaded from host memory, locate + every extract window (or "
                   "every list window) with all outputs downloaded into pageable host buffers. gather_kernel_ms and "
                   "d2h_ms: device time summed over one more pass under torch.profiler. gather_share_of_hbm counts 2 "
                   "bytes of HBM traffic per output byte (one read of the text, one write) against 7.7 TB/s: the "
                   "gather is bound by HBM bandwidth. old_path: device locate + hits, then one numpy slice of the "
                   "memory-mapped text section per hit, on the first hits of the workload",
           "check": {"ok": ok}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
