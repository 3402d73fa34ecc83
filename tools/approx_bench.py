#!/usr/bin/env python
"""Search with mismatches on a `.sufr` file on the GPU, measured (sufr_b200_index_approx), against the old way.

    python tools/approx_bench.py [--bases 1000000000] [--index-bits 32] [--queries 100000] [--reads 10000]
                                 [--out profiles/approx_bench_1000Mbp_u32.json]

1. Writes the synthetic genome of bench.py (bench.record_layout + sufr_b200_synth_dna) with `create` to a file on a
   RAM disk (/dev/shm when present) and opens it into a device index (SufrIndex.open), as tools/kmer_bench.py does.
2. Workloads: --queries 20-mers sampled from the genome (records only) with 0-3 random substitutions each, at
   k = 0, 1, 2, 3; and --reads 100-base reads sampled the same way with 0-4 substitutions, at k = 4.  For each: best of
   --reps after a warm-up, host clock around the call (it ends in a device synchronise): queries/s, matches, hits.
   Kernel time of one call from torch.profiler in a pass of its own, and the nodes and binary-search steps per depth
   (sufr_b200_index_approx_levels).
3. Baseline, the old way: every Hamming neighbour of each query over the text's non-separator bytes, enumerated on the
   host and sent through sufr_b200_index_locate in batches, on a sample of --baseline-queries 20-mers per k.  Its
   match sets (rank ranges with their mismatches) must equal the new call's on that sample.
4. Spot check: a numpy sliding window over the whole text for a few queries at k = 3 (rule (c) applied to its
   candidates, indexed positions from an exact locate of each candidate string) equals the device's hits.
Prints one JSON line with the GPU's name and power limit read in the same run, and writes it to --out."""
import argparse
import ctypes as C
import json
import os
import shutil
import sys
import tempfile
import time
from itertools import combinations, product
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import torch  # noqa: E402
import bench  # noqa: E402
import sufr_b200 as S  # noqa: E402
from sufr_b200 import _lib  # noqa: E402
from kmer_bench import best, check, gpu_identity, kernel_ms  # noqa: E402


def sample_queries(text, starts, count, length, max_subs, rng):
    """`count` windows of `length` bytes inside one record, each with 0..max_subs random ACGT substitutions."""
    n = len(text)
    ends = list(starts[1:]) + [n]
    st = np.asarray(starts, np.int64)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    out = []
    while len(out) < count:
        p = rng.integers(0, n - length, count)
        r = np.searchsorted(st, p, side="right") - 1
        ok = p + length < np.asarray(ends, np.int64)[r]
        for q in p[ok].tolist():
            w = np.frombuffer(text[q:q + length], np.uint8).copy()
            e = int(rng.integers(0, max_subs + 1))
            for j in rng.choice(length, e, replace=False):
                w[j] = acgt[(int(np.flatnonzero(acgt == w[j])[0]) + 1) % 4] if w[j] in acgt else acgt[0]
            out.append(w.tobytes())
            if len(out) == count:
                break
    return out


def neighbours(q, k, alphabet):
    """Every string within k substitutions of q over `alphabet`, with its distance."""
    out = []
    for e in range(k + 1):
        for where in combinations(range(len(q)), e):
            for subs in product(*[[b for b in alphabet if b != q[j]] for j in where]):
                w = bytearray(q)
                for j, b in zip(where, subs):
                    w[j] = b
                out.append((bytes(w), e))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=1_000_000_000)
    ap.add_argument("--index-bits", type=int, default=32, choices=[32, 64])
    ap.add_argument("--queries", type=int, default=100_000)
    ap.add_argument("--reads", type=int, default=10_000)
    ap.add_argument("--baseline-queries", type=int, default=20)
    ap.add_argument("--spot-queries", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out", default=None, help="default: profiles/approx_bench_<Mbp>Mbp_u<bits>.json")
    a = ap.parse_args()
    out_path = a.out or str(ROOT / "profiles" / f"approx_bench_{a.bases // 1_000_000}Mbp_u{a.index_bits}.json")
    gpu = gpu_identity()
    text_len, starts = bench.record_layout(a.bases)
    names = [f"chr{i + 1}" for i in range(len(starts))]
    st = np.asarray(starts, dtype=np.uint64)
    ctx = S.Context(0)
    d_text = torch.empty(text_len, dtype=torch.uint8, device="cuda")
    check(_lib.lib().sufr_b200_synth_dna(ctx.handle, d_text.data_ptr(), text_len, bench.SEED, st.ctypes.data, len(st),
                                         ord("%")))
    tmpdir = tempfile.mkdtemp(prefix="sufr_approx_", dir=a.dir)
    path = os.path.join(tmpdir, "genome.sufr")
    L = _lib.lib()
    rng = np.random.default_rng(5)
    result = {"workload": {"bases": a.bases, "text_len": text_len, "records": len(starts), "index_bits": a.index_bits,
                           "file_dir": a.dir, "queries": a.queries, "reads": a.reads, "reps": a.reps,
                           "baseline_queries": a.baseline_queries},
              "gpu": gpu, "runs": {}}
    try:
        cargs = S.SufrBuilderArgs(text=d_text.cpu().numpy().tobytes(), path=path, is_dna=True, sequence_starts=starts,
                                  sequence_names=names)
        S.create_multi(cargs, [0], index_bits=a.index_bits)
        del cargs, d_text
        torch.cuda.empty_cache()
        idx = S.SufrIndex.open(path, ctx=ctx)
        text = idx.string_at(0)
        result["workload"]["suffixes"] = idx._s
        sep = {text[-1]} | {text[c - 1] for c in starts if c > 0}
        alphabet = sorted(set(np.unique(np.frombuffer(text, np.uint8)).tolist()) - sep)
        result["workload"]["alphabet"] = bytes(alphabet).decode()
        twenty = sample_queries(text, starts, a.queries, 20, 3, rng)
        reads = sample_queries(text, starts, a.reads, 100, 4, rng)

        def approx(qs, k):
            blob, offs = idx._pack_queries(qs)
            mo = np.zeros(len(qs) + 1, np.uint64)
            hits = C.c_uint64()
            fn = lambda: check(L.sufr_b200_index_approx(idx._h, blob.ctypes.data, offs.ctypes.data, len(qs), k,  # noqa
                                                        mo.ctypes.data, C.byref(hits)))
            return fn, mo, hits

        for label, qs, k in [(f"20mer_k{k}", twenty, k) for k in range(4)] + [("100mer_k4", reads, 4)]:
            fn, mo, hits = approx(qs, k)
            t = best(fn, a.reps)
            nodes, steps = idx.approx_levels()
            kern = kernel_ms(fn)
            result["runs"][label] = {"k": k, "queries": len(qs), "query_len": len(qs[0]), "seconds": t,
                                     "queries_per_s": len(qs) / t, "matches": int(mo[-1]), "hits": int(hits.value),
                                     "kernel_ms": kern, "nodes_per_depth": nodes.tolist(),
                                     "steps_per_depth": steps.tolist(), "nodes": int(nodes.sum()),
                                     "steps": int(steps.sum())}
            print(label, json.dumps({x: y for x, y in result["runs"][label].items() if "depth" not in x}), flush=True)

        # ---- baseline: host enumeration of the neighbours, through index_locate
        base = {}
        for k in (1, 2, 3):
            sample = twenty[:a.baseline_queries]
            t0 = time.perf_counter()
            old = []
            for q in sample:
                nb = neighbours(q, k, alphabet)
                b, e, _ = idx.locate_ranges([w for w, _ in nb])
                old.append(sorted((d, int(x), int(y)) for (w, d), x, y in zip(nb, b.tolist(), e.tolist())
                                  if x != 0xFFFFFFFFFFFFFFFF))
            t_old = time.perf_counter() - t0
            t0 = time.perf_counter()
            new = idx.approx_matches(sample, k)
            t_new = time.perf_counter() - t0
            same = [sorted(r) for r in new] == old
            base[f"k{k}"] = {"queries": len(sample), "strings_per_query": len(neighbours(sample[0], k, alphabet)),
                             "old_s": t_old, "new_s": t_new, "speedup": t_old / t_new, "same_matches": same}
            print("baseline", k, json.dumps(base[f"k{k}"]), flush=True)
            assert same, f"the neighbour enumeration and index_approx differ at k = {k}"
        result["baseline"] = base

        # ---- spot check: numpy sliding window over the whole text
        t = np.frombuffer(text, np.uint8)
        n, spot = len(t), []
        for q in twenty[:a.spot_queries]:
            k, m = 3, len(q)
            qa = np.frombuffer(q, np.uint8)
            mis = np.zeros(n - m + 1, np.uint8)
            for j in range(m):
                mis += t[j:n - m + 1 + j] != qa[j]
            cand = np.flatnonzero(mis <= k)
            ok = [p for p in cand.tolist()
                  if not any(text[p + j] != q[j] and text[p + j] in sep for j in range(m))]
            words = sorted({text[p:p + m] for p in ok})
            b, e, ho = idx.locate_ranges(words)
            want = sorted(idx.hits(0, int(ho[-1]))[0].tolist())
            got = sorted(h[0] for _, hits in idx.locate_approx([q], k)[0] for h in hits)
            spot.append({"candidates": len(ok), "hits": len(got), "equal": got == want})
            assert got == want, "numpy sliding window and index_approx differ"
        result["spot_check"] = spot
        idx.close()
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    Path(out_path).parent.mkdir(parents=True, exist_ok=True)
    Path(out_path).write_text(line + "\n")


if __name__ == "__main__":
    main()
