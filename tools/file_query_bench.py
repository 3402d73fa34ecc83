#!/usr/bin/env python
"""Queries on a `.sufr` FILE, measured: open the file into a device index (sufr_b200_index_open), then batched locate on
the device (sufr_b200_index_locate + windowed sufr_b200_index_hits; mirrors SufrFile::read + SufrFile::locate,
sufr_file.rs:145-275, :1132-1169).

    python tools/file_query_bench.py [--bases 1000000000] [--index-bits 32] [--queries 4000000] [--short-queries 100000]
    python tools/file_query_bench.py --bases 3100000000 --index-bits 64

1. Writes the synthetic genome of bench.py (bench.record_layout + sufr_b200_synth_dna) with `create` to a file on a
   RAM disk (/dev/shm when present), so that the open measures the reader, not a disk.
2. Times SufrIndex.open (header check, parallel pread -> pinned slots -> device, suffix-array bound check) with a host
   clock; the call ends in a device synchronise.  Reports file bytes/s.
3. Runs 24-mers (substrings of the text: mostly one hit each) and 8-mers (thousands of hits each) through locate +
   every hit window, host buffers in and out, best of --reps.  Reports queries/s and hits/s.
4. Checks: every rank range equals that of a SufrIndex over a device build of the same text; hit windows equal a
   numpy restatement (suffix array gather + searchsorted over the sequence starts).
5. Times the per-query Python locate this replaced (one suffix copy per query + bisect) on a slice, for the speed-up.
Prints one JSON line with the GPU's name and power limit read in the same run."""
import argparse
import bisect
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


def blob_of(q):
    """(n, L) uint8 tensor -> concatenated bytes + offsets"""
    n, L = q.shape
    return q.cpu().numpy().reshape(-1).copy(), np.arange(n + 1, dtype=np.uint64) * L


class Runner:
    """locate + every hit window through the C ABI with preallocated host buffers."""

    def __init__(self, idx, window):
        self.idx, self.window = idx, window
        self.suf = np.zeros(window, np.uint64)
        self.seq = np.zeros(window, np.uint64)
        self.pos = np.zeros(window, np.uint64)

    def locate(self, blob, offs):
        nq = len(offs) - 1
        b, e, ho = np.zeros(nq, np.uint64), np.zeros(nq, np.uint64), np.zeros(nq + 1, np.uint64)
        rc = _lib.lib().sufr_b200_index_locate(self.idx._h, blob.ctypes.data, offs.ctypes.data, nq, 0, 0, 1,
                                               b.ctypes.data, e.ctypes.data, ho.ctypes.data)
        assert rc == 0, _lib.lib().sufr_b200_last_error()
        return b, e, ho

    def hits(self, first, count):
        rc = _lib.lib().sufr_b200_index_hits(self.idx._h, first, count, self.suf.ctypes.data, self.seq.ctypes.data,
                                             self.pos.ctypes.data)
        assert rc == 0, _lib.lib().sufr_b200_last_error()
        return self.suf[:count], self.seq[:count], self.pos[:count]

    def run(self, blob, offs, check=None):
        b, e, ho = self.locate(blob, offs)
        total = int(ho[-1])
        for first in range(0, total, self.window):
            n = min(self.window, total - first)
            out = self.hits(first, n)
            if check:
                check(first, out)
        return b, e, ho


def old_locate(idx, queries, starts, names):
    """The per-query Python locate this change replaced (one device->host copy per query, bisect per hit)."""
    out = []
    for r in idx.search(queries, None, True):
        hits = []
        if r is not None:
            for k, suf in enumerate(idx.suffixes(r[0], r[1] - r[0]).tolist()):
                i = bisect.bisect_right(starts, suf) - 1
                hits.append((r[0] + k, suf, names[i], suf - starts[i]))
        out.append(hits)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=1_000_000_000)
    ap.add_argument("--index-bits", type=int, default=32, choices=[32, 64])
    ap.add_argument("--queries", type=int, default=4_000_000)
    ap.add_argument("--short-queries", type=int, default=100_000)
    ap.add_argument("--window", type=int, default=1 << 26)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--old-queries", type=int, default=20_000)
    ap.add_argument("--old-short-queries", type=int, default=20)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    a = ap.parse_args()
    gpu = gpu_identity()
    text_len, starts = bench.record_layout(a.bases)
    names = [f"chr{i + 1}" for i in range(len(starts))]
    st = np.asarray(starts, dtype=np.uint64)
    ctx = S.Context(0)
    d_text = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    assert _lib.lib().sufr_b200_synth_dna(ctx.handle, d_text.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                          ord("%")) == 0

    # queries: 24-mers and 8-mers at random text positions (a few cross a record delimiter)
    g = torch.Generator(device="cuda").manual_seed(11)

    def substrings(n, L):
        p = torch.randint(0, text_len - L - 1, (n,), device="cuda", generator=g)
        return d_text[p[:, None] + torch.arange(L, device="cuda")[None, :]].contiguous()

    long_blob, long_offs = blob_of(substrings(a.queries, 24))
    short_blob, short_offs = blob_of(substrings(a.short_queries, 8))

    # ---- 1. the file
    tmpdir = tempfile.mkdtemp(prefix="sufr_file_query_", dir=a.dir)
    path = os.path.join(tmpdir, "genome.sufr")
    try:
        cargs = S.SufrBuilderArgs(text=d_text.cpu().numpy().tobytes(), path=path, is_dna=True, sequence_starts=starts,
                                  sequence_names=names)
        t0 = time.perf_counter()
        S.create_multi(cargs, [0], index_bits=a.index_bits)
        create_s = time.perf_counter() - t0
        del cargs
        file_bytes = os.path.getsize(path)

        # ---- reference answers: an index over a device build of the same text
        bargs = S.SufrBuilderArgs(text=b"", is_dna=True, sequence_starts=starts, sequence_names=names)
        r = S.build(bargs, index_bits=a.index_bits, ctx=ctx, result_memory=S.MEM_DEVICE,
                    device_text=(d_text.data_ptr(), text_len))
        built = S.SufrIndex(r, bargs)
        ref = {}
        for key, (blob, offs) in (("long", (long_blob, long_offs)), ("short", (short_blob, short_offs))):
            b, e, ho = Runner(built, 1).locate(blob, offs)
            ref[key] = (b, e, ho)
        sa_host = r.sa_tensor().cpu().numpy().view(np.uint32 if a.index_bits == 32 else np.uint64).astype(np.uint64)
        # ---- 5. the old path on a slice (over the same device index)
        lq = [bytes(long_blob[24 * i:24 * i + 24]) for i in range(min(a.old_queries, a.queries))]
        sq = [bytes(short_blob[8 * i:8 * i + 8]) for i in range(min(a.old_short_queries, a.short_queries))]
        old = {}
        for key, qs in (("long", lq), ("short", sq)):
            t0 = time.perf_counter()
            res = old_locate(built, qs, starts, names)
            dt = time.perf_counter() - t0
            old[key] = {"queries": len(qs), "hits": sum(len(h) for h in res), "s": dt}
        built.close()
        r.free()
        del d_text
        torch.cuda.empty_cache()
        ctx.trim()

        # ---- 2. open
        open_times = []
        idx = None
        for _ in range(a.reps):
            if idx is not None:
                idx.close()
                ctx.trim()
            t0 = time.perf_counter()
            idx = S.SufrIndex.open(path, ctx=ctx)
            open_times.append(time.perf_counter() - t0)
        open_s = min(open_times)

        # ---- 3. locate + hits, 4. checks
        runner = Runner(idx, a.window)
        results, ok = {}, True
        for key, (blob, offs) in (("long", (long_blob, long_offs)), ("short", (short_blob, short_offs))):
            b, e, ho = runner.run(blob, offs)  # warm-up
            same = bool(np.array_equal(b, ref[key][0]) and np.array_equal(e, ref[key][1]) and
                        np.array_equal(ho, ref[key][2]))
            total = int(ho[-1])
            # restatement of two windows: the first and one in the middle
            checked, bad = 0, 0
            for first in sorted({0, (total // 2) // a.window * a.window}):
                n = min(a.window, total - first)
                if n <= 0:
                    continue
                suf, seq, pos = runner.hits(first, n)
                h = np.arange(first, first + n, dtype=np.uint64)
                q = np.searchsorted(ho, h, side="right") - 1
                rank = b[q] + (h - ho[q])
                want_suf = sa_host[rank.astype(np.int64)]
                want_seq = np.searchsorted(st, want_suf, side="right") - 1
                bad += int((suf != want_suf).sum() + (seq != want_seq.astype(np.uint64)).sum() +
                           (pos != want_suf - st[want_seq]).sum())
                checked += n
            times = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                runner.run(blob, offs)
                times.append(time.perf_counter() - t0)
            dt = min(times)
            nq = len(offs) - 1
            found = int((b != NONE).sum())
            results[key] = {"queries": nq, "query_len": int(offs[1]), "found": found, "hits": total,
                            "s": dt, "queries_per_s": nq / dt, "hits_per_s": total / dt,
                            "ranges_identical_to_build_index": same, "hits_checked": checked, "hits_bad": bad,
                            "old_path": old[key],
                            "speedup_vs_old_path": (nq / dt) / (old[key]["queries"] / old[key]["s"])}
            ok = ok and same and bad == 0
        info = idx.info
        idx.close()
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    out = {"metric": "file open bytes/s; locate queries/s and hits/s (device locate + windowed hits)",
           "gpu": gpu, "bases": a.bases, "text_len": text_len, "index_bits": a.index_bits,
           "num_suffixes": info["num_suffixes"], "records": len(starts), "file_bytes": file_bytes,
           "file_dir": a.dir, "create_s": create_s,
           "open": {"s": open_s, "all_s": open_times, "bytes_per_s": file_bytes / open_s,
                    "note": "host clock around SufrIndex.open (ends in a device synchronise); the file was just "
                            "written, so it is read from page cache / RAM disk"},
           "locate": results, "window": a.window, "reps": a.reps,
           "note": "timed region: queries uploaded from host memory, search + hit-offset scan, every hit window "
                   "(suffix, sequence, position) downloaded to host memory; best of reps. old_path: the per-query "
                   "Python locate it replaced, on the first queries of each batch",
           "check": {"ok": ok}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
