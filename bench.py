#!/usr/bin/env python
"""bench.py -- suffixes/second of SA+LCP construction (BASELINE.json metric) on B200.

A "step" is one complete build (encode -> keys -> sort -> refine -> LCP -> finish) of the synthetic
3.1 Gbp DNA text of BASELINE.json configs[1] (24 records with chromosome-proportional lengths, iid
uniform ACGT, '%' between records, '$' at the end; u64 SA/LCP as the config names).

  value : text already resident in HBM, SA/LCP left in HBM (device-timed, whole job over all ranks)
  e2e   : the same build through the C ABI with HOST buffers -- pinned text copied H2D, SA/LCP/text
          copied D2H -- all inside the timed region
  roofline     : the dominant kernel (radix-sort scatter pass), CUDA-event timed per launch inside the step
  cpu_baseline : the oracle restatement of the reference's rayon path on a bounded prefix of the same text
  verify       : FULL on-device check of the last timed result (sufr_b200_verify): every SA entry indexed and
                 unique, every adjacent pair in order, every LCP exact -- pairs = num_suffixes - 1
  configs      : the other BASELINE.json configs (1, 3, 4, 5 and the repetitive variant 2b) at their full sizes
                 on one GPU, each with its own value, job roofline and full verification (--no-configs to skip)

`--dump-outputs DIR` writes what the last timed step returned (see write_outputs), so that two builds of the project
can be compared output for output: the workload text is generated from a fixed seed, so equal arguments give equal
inputs.

`--impl reference` times the reference's CPU algorithm (oracle port; the Rust reference cannot be compiled
in this image) with the flags the workload names (-n 16, u64 indices) on a bounded sample of the same
workload; the sample size is part of `config` in BOTH arms (reference_arm_sample_bases).

N > 1 (torchrun): the text is replicated, rank r builds key-range shard r (no data-path collective), one
all_gather of (count, first, last) repairs the seam LCPs.  Fixed total work => "scaling": "strong".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# human chromosome lengths (Mbp, GRCh38 1..22, X, Y): only the proportions matter
CHROM_MBP = [248, 242, 198, 190, 182, 171, 159, 145, 138, 134, 135, 133, 114, 107, 102, 90, 83, 80, 59, 64, 47, 51,
             156, 57]
SEED = 2  # SURVEY.md section 8(d), config 2


def record_layout(total_bases: int):
    """24 record lengths proportional to the human chromosomes, summing to total_bases; returns
    (text_len, record_starts) with one delimiter between records and the trailing '$'."""
    tot = sum(CHROM_MBP)
    lens = [max(1, total_bases * c // tot) for c in CHROM_MBP]
    lens[0] += total_bases - sum(lens)
    starts, pos = [], 0
    for ln in lens:
        starts.append(pos)
        pos += ln + 1  # delimiter (or the final '$')
    return pos, starts


def synth_prefix_numpy(n: int, text_len: int, starts, seed: int = SEED) -> bytes:
    """CPU restatement of synth_dna_kernel / synth_marks_kernel for the first n bytes of the text."""
    i = np.arange(1, n + 1, dtype=np.uint64)
    c = np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) * c + i * c
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    out = np.frombuffer(b"ACGT", dtype=np.uint8)[(z >> np.uint64(62)).astype(np.int64)].copy()
    for s in starts[1:]:
        if 1 <= s <= n:
            out[s - 1] = ord("%")
    if n == text_len:
        out[n - 1] = ord("$")
    return out.tobytes()


class ClockSampler:
    """Samples SM clocks / throttle reasons while the timed region runs (B200_PROFILING.md): through NVML every
    10 ms when pynvml is importable (a multi-GPU timed region lasts ~150 ms), else through nvidia-smi."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    BITS = [0x8, 0x40, 0x20, 0x4]  # nvmlClocksEventReason{HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap}

    def __init__(self, index: int, uuid: str = None):
        self.index, self.uuid = index, uuid
        self.samples, self._stop, self._t = [], threading.Event(), None  # [sm, sm_max, watts, 4 x "Active"/"Not Active"]
        self.source = "nvidia-smi"

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        if self.uuid:
            try:
                return pynvml, pynvml.nvmlDeviceGetHandleByUUID(self.uuid if self.uuid.startswith("GPU-") else "GPU-" + self.uuid)
            except Exception:
                pass
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _run(self):
        try:
            nv, h = self._nvml_handle()
            sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.source = "nvml"
            while not self._stop.is_set():
                mask = reasons_fn(h)
                self.samples.append([nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), sm_max, nv.nvmlDeviceGetPowerUsage(h) / 1000.0]
                                    + ["Active" if mask & b else "Not Active" for b in self.BITS])
                self._stop.wait(0.01)
            return
        except Exception:
            if self.samples:
                return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = [nm for k, nm in enumerate(self.NAMES) if any(str(s[3 + k]).lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(float(s[2]) for s in self.samples), "source": self.source}


def oracle_run(sample: bytes, threads: int, partitions: int, index_bits: int = 64):
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle as O
    t0 = time.perf_counter()
    r = O.oracle_build(sample, is_dna=True, num_partitions=partitions, threads=threads, index_bits=index_bits)
    dt = time.perf_counter() - t0
    return r, dt


DUMP_SAMPLE = 1 << 20  # entries per dumped array: about 38 MB in all
DUMP_SEED = 20261020


def dump_sample(n: int, seed: int) -> np.ndarray:
    """Sorted, seeded sample of range(n), a function of (n, seed) only; all of range(n) when n <= DUMP_SAMPLE."""
    if n <= DUMP_SAMPLE:
        return np.arange(n, dtype=np.int64)
    return np.unique(np.random.default_rng(seed).integers(0, n, DUMP_SAMPLE, dtype=np.int64))


def write_outputs(out_dir, total_suffixes, ranks, sa, lcp, text_len, positions, text):
    """--dump-outputs: sizes.npy = [suffixes, text bytes]; sa.npy / lcp.npy = the suffix and LCP arrays at the sampled
    ranks (ranks.npy); text.npy = the transformed text at the sampled positions (positions.npy).  Indices are float64
    (exact below 2^53), text bytes float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("sizes", [total_suffixes, text_len]), ("ranks", ranks), ("sa", sa), ("lcp", lcp),
                    ("positions", positions)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))
    np.save(os.path.join(out_dir, "text.npy"), np.asarray(text, dtype=np.float32))


def dump_device_result(out_dir, res, rank, world, dev):
    """write_outputs for a device result; with N > 1 every rank reads the sampled ranks of its shard and rank 0
    writes them."""
    import torch
    import torch.distributed as dist
    ranks = dump_sample(res.total_suffixes, DUMP_SEED)
    lo = res.shard_offset
    idx = torch.from_numpy(ranks[(ranks >= lo) & (ranks < lo + res.num_suffixes)] - lo).to(dev)

    def read(t):
        t = t[idx].to(torch.int64)
        return (t & 0xFFFFFFFF if res.index_bits == 32 else t).cpu().numpy()  # u32 read through an int32 view
    parts = [(read(res.sa_tensor()), read(res.lcp_tensor()))]
    if world > 1:
        mine, parts = parts[0], [None] * world
        dist.all_gather_object(parts, mine)
    if rank == 0:
        positions = dump_sample(res.text_len, DUMP_SEED + 1)
        text = res.text_tensor()[torch.from_numpy(positions).to(dev)].cpu().numpy()
        write_outputs(out_dir, res.total_suffixes, ranks, np.concatenate([p[0] for p in parts]),
                      np.concatenate([p[1] for p in parts]), res.text_len, positions, text)


def reference_sample_bases(args):
    """Bases per step of the reference arm: bounded so that (steps + warmup) builds end within a few minutes
    at the ~25 M suffixes/s the port reaches, at most 1 Gbp."""
    if args.cpu_sample:
        return min(args.cpu_sample, args.bases)
    budget_s, rate = 200.0, 25e6
    per_step = int(budget_s * rate / max(1, args.steps + args.warmup))
    return int(max(32_000_000, min(1_000_000_000, per_step, args.bases)))


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (oracle port) on the box's host cores, flags as the workload
    names them (-n 16, u64 SA / LCP)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    text_len, starts = record_layout(args.bases)
    sample_n = reference_sample_bases(args)
    sample = synth_prefix_numpy(sample_n, text_len, starts)
    if sample_n < text_len:
        sample = sample[:-1] + b"$"
    for _ in range(args.warmup):
        oracle_run(sample, cores, 16, args.index_bits)
    t = 0.0
    nsuf = 0
    for _ in range(args.steps):
        r, dt = oracle_run(sample, cores, 16, args.index_bits)
        t += dt
        nsuf += r.num_suffixes
    value = nsuf / t
    if args.dump_outputs:
        ranks, positions = dump_sample(r.num_suffixes, DUMP_SEED), dump_sample(len(r.text), DUMP_SEED + 1)
        write_outputs(args.dump_outputs, r.num_suffixes, ranks, r.sa[ranks], r.lcp[ranks], len(r.text), positions,
                      np.frombuffer(r.text, dtype=np.uint8)[positions])
    line = {
        "impl": "reference", "metric": "suffixes/sec (SA+LCP)", "value": value, "unit": "suffixes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, text_len),
        "cpu_baseline": {"value": value, "unit": "suffixes/s", "cores": cores, "kind": "port",
                         "sample": f"every step builds the first {sample_n} bytes of the workload text "
                                   f"(u{args.index_bits} indices, -n 16 as the workload names it: the sort phase runs "
                                   f"16 partitions in parallel), oracle restatement of sufr_builder.rs with {cores} "
                                   f"threads, partitions kept in RAM"},
        "e2e": {"value": value, "unit": "suffixes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, text_len):
    return {"workload": f"sufr create --dna, {args.bases} bp synthetic iid ACGT in 24 records (BASELINE configs[1]), "
                        f"u{args.index_bits} SA+LCP", "text_len": text_len, "index_bits": args.index_bits,
            "flags": "--dna -n 16", "seed": SEED, "reference_arm_sample_bases": reference_sample_bases(args),
            "l2_policy": "inputs (>= 3 GB text, >= 37 GB key/position arrays) are far larger than the 126 MB L2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bases", type=int, default=3_100_000_000)
    ap.add_argument("--index-bits", type=int, default=64, choices=[32, 64])
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="bases per step of the reference arm (0 = as many as fit ~200 s over steps + warmup, <= 1 Gbp)")
    ap.add_argument("--cpu-baseline-sample", type=int, default=400_000_000,
                    help="bases of the one cpu_baseline build inside our own arm (about 15-20 s of CPU work)")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs (1, 3, 4, 5, 2b)")
    ap.add_argument("--no-e2e-file", action="store_true", help="skip the host text -> .sufr file figure")
    ap.add_argument("--configs", default="config1,config3,config4,config5,config2b")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--verify", type=int, default=1, help="0 = skip the full on-device verification of the last result")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's suffix array, LCP array and text (seeded sample) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import sufr_b200 as S
    from sufr_b200.distributed import finish_shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    text_len, starts = record_layout(args.bases)
    ctx = S.Context(local_rank)
    d_text = torch.empty(text_len, dtype=torch.uint8, device=dev)
    from sufr_b200 import _lib
    import ctypes as C
    st = np.asarray(starts, dtype=np.uint64)
    rc = _lib.lib().sufr_b200_synth_dna(ctx.handle, d_text.data_ptr(), text_len, SEED, st.ctypes.data, len(st), ord("%"))
    assert rc == 0, _lib.lib().sufr_b200_last_error()
    bargs = S.SufrBuilderArgs(text=b"", is_dna=True, num_partitions=16, sequence_starts=starts,
                              sequence_names=[f"chr{i + 1}" for i in range(len(starts))])

    def step_device():
        r = S.build(bargs, index_bits=args.index_bits, ctx=ctx, result_memory=S.MEM_DEVICE,
                    device_text=(d_text.data_ptr(), text_len), rank=rank, world_size=world)
        meta = finish_shard(r) if world > 1 else None
        return r, meta

    # ---------------- value: resident text -> resident SA/LCP
    for _ in range(args.warmup):
        step_device()[0].free()
    barrier()
    results = []
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        gpu_uuid = None
    with ClockSampler(local_rank, gpu_uuid) as clocks:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r, last_meta = step_device()
            results.append((r.num_suffixes, r.total_suffixes, r.timings, r.kernel_launches))
            last = r
            if _ + 1 < args.steps:
                r.free()
        barrier()
        elapsed = time.perf_counter() - t0
    el = torch.tensor([elapsed], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    elapsed = float(el.item())
    total_suffixes = results[-1][1]
    value = total_suffixes * args.steps / elapsed
    tm = results[-1][2]
    launches = sum(x[3] for x in results)

    # ---------------- FULL verification of the last timed result on the device (outside the timed region)
    verify = verify_full(last, last_meta, rank, world, dev) if args.verify else None
    if args.dump_outputs:
        dump_device_result(args.dump_outputs, last, rank, world, dev)
    last.free()

    # ---------------- e2e: host text in, host SA/LCP out, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, S, ctx, d_text, text_len, bargs, rank, world, dev, barrier)

    # ---------------- e2e_file: host text in, one `.sufr` file out (sufr::create through the C ABI), N=1 only
    e2e_file = None
    if not args.no_e2e and not args.no_e2e_file and world == 1:
        e2e_file = run_e2e_file(args, S, ctx, d_text, text_len, bargs, total_suffixes, dev)

    # ---------------- CPU baseline on a bounded prefix (rank 0, N=1 only)
    cpu = None
    if not args.no_cpu and rank == 0 and world == 1:
        cores = os.cpu_count() or 1
        sample_n = min(args.cpu_baseline_sample, text_len)
        sample = d_text[:sample_n].cpu().numpy().tobytes()
        if sample_n < text_len:
            sample = sample[:-1] + b"$"
        r, dt = oracle_run(sample, cores, 16, args.index_bits)
        cpu = {"value": r.num_suffixes / dt, "unit": "suffixes/s", "cores": cores, "kind": "port",
               "sample": f"one build of the first {sample_n} bytes of the workload text (u{args.index_bits} indices, "
                         f"-n 16 as the workload names it); oracle restatement of sufr_builder.rs, {cores} threads, "
                         f"partitions in RAM; {dt:.2f} s"}
    del d_text
    torch.cuda.empty_cache()

    # ---------------- the other BASELINE configs at full size (N=1 only): value, job roofline, full verification
    configs = None
    if not args.no_configs and world == 1:
        configs = run_configs(args, S, ctx, dev)
    variants = {"repetitive": configs["config2b"]} if configs and "config2b" in configs else None

    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        dk_ms = tm["dominant_kernel_ms"] / max(1, tm["dominant_kernel_launches"])
        achieved = tm["dominant_kernel_bytes"] / (dk_ms * 1e-3) / 1e9 if dk_ms > 0 else 0.0
        w = args.index_bits // 8
        job_bytes = text_len + 2 * total_suffixes * w
        line = {
            "metric": "suffixes/sec (SA+LCP)", "value": value, "unit": "suffixes/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64" if args.index_bits == 64 else "u32", "data": "synthetic",
            "config": workload_config(args, text_len),
            "clocks": clocks.summary(),
            "e2e": e2e, "e2e_file": e2e_file, "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "osort::onesweep_kernel<u64,u32,512,16> = radix scatter pass of the main sort",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650 GB/s",
                         "traffic": traffic_estimate(tm["dominant_kernel_bytes"]), "traffic_source": TRAFFIC_SOURCE,
                         "algorithmic_bytes": tm["dominant_kernel_bytes"], "launch_ms": dk_ms, "launches_per_step": tm["dominant_kernel_launches"],
                         "share_of_step": tm["dominant_kernel_ms"] / (1e3 * elapsed / args.steps),
                         "job": {"algorithmic_bytes": job_bytes,
                                 "achieved": job_bytes * args.steps / elapsed / 1e9 / world,
                                 "frac": job_bytes * args.steps / elapsed / 1e9 / world / peak,
                                 "note": "A = n + 2*s*sizeof(T) per SURVEY 8(d), per GPU"}},
            "cpu_baseline": cpu,
            "configs": configs,
            "variants": variants,
            "phases_ms": {k: v for k, v in tm.items() if k.endswith("_ms")},
            "verify": verify,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


TRAFFIC_SOURCE = ("dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel on the "
                  "1.0 Gbp workload (profiles/r2_v12_ncu_full_1000Mbp_build_raw.csv: 12.557 GB + 12.451 GB for "
                  "24.000 GB algorithmic), scaled to this launch's element count")


def traffic_estimate(algorithmic_bytes):
    """DRAM bytes per launch of the dominant kernel (see TRAFFIC_SOURCE)."""
    return algorithmic_bytes * (12.557185 + 12.451262) / 24.000000


FULL_SIZES = {"config1": 10_000_000, "config2b": 3_100_000_000, "config3": 1_000_000_000,
              "config4": 500_000_000, "config5": 1_000_000_000}
CONFIG_NOTES = {
    "config1": "BASELINE configs[0]: sufr create --dna -n 16, 10 Mbp iid ACGT, u32",
    "config2b": "BASELINE configs[1], repetitive variant: ~50 % of the bases are mutated copies of earlier 0.3-6 kb "
                "segments, some N / soft-masked stretches, u64",
    "config3": "BASELINE configs[2]: protein alphabet, 1 G residues in 10 000 records, --max-query-len 32, u32",
    "config4": "BASELINE configs[3]: --dna --seed-mask 1101101101 on 500 Mbp (the reference rejects the mask together "
               "with --max-query-len, so the cap is dropped), u32",
    "config5": "BASELINE configs[4]: --dna --allow-ambiguity --ignore-softmask, 1 Gbp tandem repeats / low entropy / "
               "soft-masked and N runs, u32",
}


def run_configs(args, S, ctx, dev):
    """One warm-up + two timed device-resident builds of every other BASELINE config at its full size (scaled with
    --bases when the headline is scaled), each followed by the full on-device verification."""
    import torch
    import workloads
    peak = 6650.0
    try:
        peak = float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("hbm_gbs", peak))
    except Exception:
        pass
    scale = min(1.0, args.bases / 3_100_000_000)
    out = {}
    for name in [c for c in args.configs.split(",") if c]:
        size = max(100_000, int(FULL_SIZES[name] * scale))
        t0 = time.perf_counter()
        w = workloads.ALL[name](size)
        gen_s = time.perf_counter() - t0
        t = torch.frombuffer(bytearray(w.text), dtype=torch.uint8).to(dev)
        bargs = S.SufrBuilderArgs(text=b"", sequence_starts=w.sequence_starts, sequence_names=w.sequence_names, **w.flags)
        times, info, ver = [], None, None
        for i in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = S.build(bargs, index_bits=w.index_bits, ctx=ctx, result_memory=S.MEM_DEVICE,
                        device_text=(t.data_ptr(), t.numel()))
            torch.cuda.synchronize()
            if i:
                times.append(time.perf_counter() - t0)
            info = (r.num_suffixes, int(r.c.refine_rounds), int(r.c.doubling_rounds), r.timings, r.kernel_launches)
            if i == 2 and args.verify:
                ver = r.verify()
            r.free()
        ms = 1e3 * sum(times) / len(times)
        job_bytes = t.numel() + 2 * info[0] * (w.index_bits // 8)
        out[name] = {"workload": CONFIG_NOTES[name], "text_len": t.numel(), "num_suffixes": info[0],
                     "index_bits": w.index_bits, "flags": {k: v for k, v in w.flags.items()},
                     "ms_per_step": ms, "value": info[0] / (ms * 1e-3), "unit": "suffixes/s",
                     "refine_rounds": info[1], "doubling_rounds": info[2], "gpu_launches_per_step": info[4],
                     "phases_ms": {k: v for k, v in info[3].items() if k.endswith("_ms")},
                     "roofline_job": {"algorithmic_bytes": job_bytes, "achieved": job_bytes / (ms * 1e-3) / 1e9,
                                      "frac": job_bytes / (ms * 1e-3) / 1e9 / peak, "unit": "GB/s"},
                     "verify": verify_summary(ver, info[0]) if ver else None, "generate_s": round(gen_s, 1)}
        del t
        torch.cuda.empty_cache()
        ctx.trim()
    return out


def verify_summary(rep, total_suffixes):
    """Bench-line form of a SufrB200VerifyReport."""
    errors = rep["order_errors"] + rep["lcp_errors"] + rep["out_of_range"] + rep["not_indexed"] + rep["duplicates"]
    return {"method": "sufr_b200_verify: every SA entry indexed + unique (bitmap), every adjacent pair compared on the "
                      "text bytes (order + exact LCP)",
            "pairs": rep["pairs_checked"], "mismatches": rep["order_errors"] + rep["lcp_errors"],
            "order_errors": rep["order_errors"], "lcp_errors": rep["lcp_errors"],
            "position_errors": rep["out_of_range"] + rep["not_indexed"] + rep["duplicates"],
            "suffixes": total_suffixes, "expected_suffixes": rep["expected_suffixes"],
            "count_ok": rep["expected_suffixes"] == total_suffixes, "max_lcp": rep["max_lcp"],
            "ok": errors == 0 and rep["expected_suffixes"] == total_suffixes, "ms": rep["ms"]}


def verify_full(res, meta, rank, world, dev):
    """Full verification of the last timed result: every rank checks its shard (with the seam pair), the error
    counters are summed over the ranks."""
    import torch
    import torch.distributed as dist
    from sufr_b200.distributed import previous_last_suffix
    prev = previous_last_suffix(meta, rank) if (world > 1 and meta) else None
    rep = res.verify(prev if res.num_suffixes else None)
    keys = ["pairs_checked", "order_errors", "lcp_errors", "out_of_range", "not_indexed", "duplicates", "lcp_sum"]
    vals = torch.tensor([rep[k] for k in keys] + [res.num_suffixes], dtype=torch.int64, device=dev)
    mx = torch.tensor([rep["max_lcp"], int(rep["ms"] * 1000)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    tot = {k: int(v) for k, v in zip(keys, vals.tolist()[:-1])}
    tot.update(expected_suffixes=rep["expected_suffixes"], max_lcp=int(mx[0].item()), ms=mx[1].item() / 1000.0)
    return verify_summary(tot, int(vals[-1].item()))


def run_e2e(args, S, ctx, d_text, text_len, bargs, rank, world, dev, barrier):
    import torch
    import torch.distributed as dist
    from sufr_b200.distributed import finish_shard
    h_text = torch.empty(text_len, dtype=torch.uint8, pin_memory=True) if rank == 0 or world == 1 else None
    if h_text is not None:
        h_text.copy_(d_text)
    torch.cuda.synchronize()
    staging = torch.empty(text_len, dtype=torch.uint8, device=dev) if world > 1 else None

    def step():
        if world == 1:
            return S.build(_with_text(bargs, h_text), index_bits=args.index_bits, ctx=ctx,
                           result_memory=S.MEM_HOST)
        # N > 1: rank 0 uploads, NCCL broadcast replicates the text, every rank builds and downloads its shard
        if rank == 0:
            staging.copy_(h_text, non_blocking=True)
        dist.broadcast(staging, src=0)
        torch.cuda.synchronize()
        r = S.build(bargs, index_bits=args.index_bits, ctx=ctx, result_memory=S.MEM_HOST,
                    device_text=(staging.data_ptr(), text_len), rank=rank, world_size=world)
        finish_shard(r)
        return r

    step().free()  # warm-up: page-locks the result buffers once
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    h2d = 0
    out_bytes = 0
    tot = 0
    for _ in range(args.e2e_steps):
        r = step()
        d2h = r.d2h_bytes                      # bytes that crossed PCIe (compact encoding, see sufr_b200.h)
        h2d = r.h2d_bytes if world == 1 else (text_len if rank == 0 else 0)
        out_bytes = (r.text_len if rank == 0 else 0) + 2 * r.num_suffixes * (args.index_bits // 8)
        tot = r.total_suffixes
        _ = int(r.sa[:1024].sum()) if r.num_suffixes else 0  # read the step's result on the host
        r.free()
    barrier()
    elapsed = time.perf_counter() - t0
    el = torch.tensor([elapsed], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    elapsed = float(el.item())
    return {"value": tot * args.e2e_steps / elapsed, "unit": "suffixes/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "host_result_bytes_per_step": out_bytes,
            "ms_per_step": 1e3 * elapsed / args.e2e_steps, "steps": args.e2e_steps,
            "note": "pinned host text -> H2D -> build -> D2H (LCP as bytes + exceptions, u64 SA as u32, widened by host "
                    "threads into the pinned u64 result arrays), per step; bytes are those of rank 0"}


def run_e2e_file(args, S, ctx, d_text, text_len, bargs, total_suffixes, dev):
    """Host text -> one `.sufr` file on a RAM disk, through sufr_b200_create_multi (what `sufr-b200 create` calls):
    upload, build, and the file written straight from device memory by the streaming writer.  One run (the file
    is new every time, as for a user); skipped when the box cannot hold the file in RAM."""
    import copy
    import shutil
    import torch
    w = args.index_bits // 8
    file_bytes = text_len + 2 * total_suffixes * w + 4096
    h = d_text.cpu().numpy()
    torch.cuda.synchronize()
    ctx.trim()  # the call below works in a context of its own: give the pooled device and pinned memory back first
    torch.cuda.empty_cache()
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 0
    shm_free = shutil.disk_usage("/dev/shm").free if os.path.isdir("/dev/shm") else 0
    if avail < file_bytes * 1.2 + text_len + (8 << 30) or shm_free < file_bytes * 1.05:
        return {"skipped": f"needs {file_bytes / 1e9:.1f} GB of RAM disk; available RAM {avail / 1e9:.1f} GB, "
                           f"/dev/shm free {shm_free / 1e9:.1f} GB"}
    path = f"/dev/shm/sufr_b200_bench_{os.getpid()}.sufr"
    b = copy.copy(bargs)
    b.text = memoryview(h)
    b.path = path
    try:
        t0 = time.perf_counter()
        res = S.create_multi(b, [dev.index or 0], args.index_bits)
        dt = time.perf_counter() - t0
        size = os.path.getsize(path)
        return {"value": res["num_suffixes"] / dt, "unit": "suffixes/s", "s": dt, "file_bytes": size, "path": "/dev/shm",
                "device_ms": res["timings"]["total_ms"], "write_ms": res["timings"].get("d2h_ms"),
                "note": "host text -> sufr_b200_create_multi on this GPU -> .sufr (version 6) on a RAM disk, one run, wall clock"}
    except Exception as e:  # an extra figure must not cost the bench line (e.g. a RAM disk that fills up)
        return {"error": f"{type(e).__name__}: {e}"[:300]}
    finally:
        try:
            os.remove(path)
        except OSError:
            pass


def _with_text(bargs, h_text):
    """SufrBuilderArgs whose text is a zero-copy view of the pinned host tensor."""
    import copy
    b = copy.copy(bargs)
    b.text = memoryview(h_text.numpy())
    return b


if __name__ == "__main__":
    main()
