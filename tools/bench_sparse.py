"""Sparse (CSR) k-mer count rows: kernel time, Gbases/s and algorithmic bytes/s of ktb_sparse_vectorise_device, next to
the dense rows of the same data where k <= 12.  Prints one JSON object and writes it to --out.

Bytes of a sparse call: sum(len) + 8 (n + 1) offsets + 8 (n + 1) row_ptr + nnz (8 + esize) codes and values.  Bytes of a
dense call: bench.algorithmic_bytes.  Share of peak = bytes / time over the measured copy peak (COPY_PEAK_GBS).
Inputs are generated on the GPU by bench.make_workload_torch (the benchmark's seeded workloads)."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

COPY_PEAK_GBS = 6462.7   # device-to-device copy peak measured on the B200 (GB/s)

# (label, bench workload, scale, k, canonical, out dtype, norm, compare with the dense path)
CASES = [
    ("reads150_k21", "reads150_k5", 1.0, 21, 1, "f32", 1, False),
    ("reads150_k31", "reads150_k5", 1.0, 31, 1, "f32", 1, False),
    ("contigs_k21", "contigs_k4", 1.0, 21, 1, "f32", 1, False),
    ("reads100k_k10", "reads100k_k10", 1.0, 10, 1, "u32", 0, True),
    ("reads100k_200_k12", "reads100k_k10_f32", 0.1, 12, 1, "f32", 1, True),
]
DT = {"u32": (0, 4), "f32": (1, 4), "f64": (2, 8)}


def gpu_identity() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = line.partition(",")
    return {"gpu": name.strip(), "power_limit": power.strip()}


def timed(torch, fn, min_seconds: float, warmup: int):
    """Mean milliseconds per call from CUDA events over at least min_seconds of back-to-back calls (after warm-up)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    steps, elapsed_ms = 0, 0.0
    t0 = time.time()
    while elapsed_ms < min_seconds * 1e3 or steps < 3:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        elapsed_ms += a.elapsed_time(b)
        steps += 1
        if time.time() - t0 > 60 * min_seconds:
            break
    return elapsed_ms / steps, steps


def device_intervals(torch, fn):
    """[(name, start_us, end_us)] of the device activities (kernels, copies) of one call of fn, from torch.profiler."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [(e.name, e.time_range.start, e.time_range.end) for e in prof.events() if e.device_type == DeviceType.CUDA]


def union_length(iv):
    total, end = 0.0, float("-inf")
    for a, b in sorted(iv):
        if b > end:
            total += b - max(a, end)
            end = b
    return total


def kernel_breakdown(iv) -> dict:
    """Device milliseconds per sparse kernel family in one call."""
    out = {}
    for name, a, b in iv:
        for fam in ("sparse_tile", "sparse_merge", "sparse_scan", "sparse_count", "sparse_write"):
            if fam in name:
                out[fam + "_ms"] = out.get(fam + "_ms", 0.0) + (b - a) / 1e3
    return out


def run_host_overlap(torch, lib):
    """The host entry point over 1 M reads of 150 bp (150 Mbp: three chunks of 2^26 bases) at k = 21 into pageable numpy
    arrays: wall time, and how long the device-to-host copies of rows ran while a kernel of another chunk ran."""
    import bench
    from kmertools_b200 import kmer_counts
    bases, offsets = bench.make_workload(bench.WORKLOADS["reads150_k5"], 0.1, bench._NP())
    bases, offsets = np.asarray(bases), np.asarray(offsets).astype(np.uint64)
    kmer_counts((bases, offsets), 21, True, 1, np.float32)   # warm-up
    t0 = time.time()
    rows = kmer_counts((bases, offsets), 21, True, 1, np.float32)
    wall = time.time() - t0
    iv = device_intervals(torch, lambda: kmer_counts((bases, offsets), 21, True, 1, np.float32))
    kern = [(a, b) for name, a, b in iv if "sparse_" in name]
    d2h = [(a, b) for name, a, b in iv if "DtoH" in name or "Device -> Pageable" in name or "Device -> Pinned" in name]
    both = union_length(kern) + union_length(d2h) - union_length(kern + d2h)
    return {"case": "host_entry_reads150_k21_1M", "n": len(offsets) - 1, "bases": int(offsets[-1]),
            "nnz": int(rows[0][-1]), "wall_ms": wall * 1e3, "gbases_s_end_to_end": int(offsets[-1]) / wall / 1e9,
            "profiled_kernel_union_ms": union_length(kern) / 1e3, "profiled_d2h_union_ms": union_length(d2h) / 1e3,
            "profiled_d2h_during_kernels_ms": both / 1e3}


def run_case(torch, lib, case, min_seconds, warmup):
    import bench
    from kmertools_b200 import OligoComputer, _lib
    from tests.sparse_ref import sparse_rows
    label, wl, scale, k, canonical, dt, norm, dense = case
    code, esize = DT[dt]
    dev = torch.device("cuda", 0)
    tb, to = bench.make_workload_torch(bench.WORKLOADS[wl], scale, dev)
    n = to.numel() - 1
    total = int(to[-1])
    stream = torch.cuda.current_stream(dev).cuda_stream
    row_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    _lib.check(lib.ktb_sparse_vectorise_device(tb.data_ptr(), to.data_ptr(), n, total, k, canonical, norm, code,
                                               row_ptr.data_ptr(), None, None, 0, None, stream))
    nnz = int(row_ptr[-1])
    codes = torch.empty(max(nnz, 1), dtype=torch.int64, device=dev)
    values = torch.empty(max(nnz, 1) * esize, dtype=torch.uint8, device=dev)

    def sparse_call():
        _lib.check(lib.ktb_sparse_vectorise_device(tb.data_ptr(), to.data_ptr(), n, total, k, canonical, norm, code,
                                                   row_ptr.data_ptr(), codes.data_ptr(), values.data_ptr(), nnz, None,
                                                   stream))
    ms, steps = timed(torch, sparse_call, min_seconds, warmup)
    breakdown = kernel_breakdown(device_intervals(torch, sparse_call))
    sbytes = total + 8 * (n + 1) + 8 * (n + 1) + nnz * (8 + esize)
    out = {"case": label, "workload": wl, "scale": scale, "k": k, "canonical": canonical, "dtype": dt, "norm": norm,
           "n": n, "bases": total, "nnz": nnz, "sparse_ms": ms, "sparse_steps": steps,
           "sparse_gbases_s": total / ms / 1e6, "sparse_bytes": sbytes, "sparse_gb_s": sbytes / ms / 1e6,
           "sparse_share_of_copy_peak": sbytes / ms / 1e6 / COPY_PEAK_GBS, "profiled_kernels": breakdown}
    # oracle parity sample: three sequences (first, middle, last) against the Python restatement
    rp = row_ptr.cpu().numpy()
    ok = True
    vdt = {0: np.uint32, 1: np.float32, 2: np.float64}[code]
    for i in (0, n // 2, n - 1):
        lo, hi = int(to[i]), int(to[i + 1])
        b = tb[lo:hi].cpu().numpy()
        w = sparse_rows(b, np.array([0, hi - lo], np.uint64), k, bool(canonical), norm)
        a0, a1 = int(rp[i]), int(rp[i + 1])
        got_c = codes[a0:a1].cpu().numpy().astype(np.uint64)
        got_v = values[a0 * esize:a1 * esize].cpu().numpy().view(vdt)
        ok &= np.array_equal(got_c, w[1]) and np.array_equal(got_v, w[2].astype(vdt))
    out["parity_sample_ok"] = bool(ok)
    del codes, values
    if dense:
        oc = OligoComputer(k)
        dim = oc.dim(bool(canonical))
        rows = torch.empty((n, dim), dtype={0: torch.int32, 1: torch.float32, 2: torch.float64}[code], device=dev)

        def dense_call():
            oc.vectorise_device(tb.data_ptr(), to.data_ptr(), n, total, rows.data_ptr(), norm_mode=norm,
                                mins=bool(canonical), out_dtype=code, stream=stream)
        dms, dsteps = timed(torch, dense_call, min_seconds, warmup)
        dbytes = bench.algorithmic_bytes(total, n, dim, esize)
        out.update(dense_ms=dms, dense_steps=dsteps, dense_gbases_s=total / dms / 1e6, dense_bytes=dbytes,
                   dense_gb_s=dbytes / dms / 1e6, dense_share_of_copy_peak=dbytes / dms / 1e6 / COPY_PEAK_GBS,
                   sparse_over_dense_time=ms / dms, output_bytes_sparse=nnz * (8 + esize) + 8 * (n + 1),
                   output_bytes_dense=n * dim * esize)
        del rows
        oc.close()
    del tb, to, row_ptr
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default="bench_sparse.json")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES) + ",host_overlap")
    args = ap.parse_args()
    import torch
    from kmertools_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse needs a CUDA device")
    lib = _lib.load()
    result = {"tool": "tools/bench_sparse.py", **gpu_identity(), "copy_peak_gb_s": COPY_PEAK_GBS,
              "min_seconds": args.min_seconds, "cases": []}
    want = set(args.cases.split(","))
    for case in CASES:
        if case[0] in want:
            r = run_case(torch, lib, case, args.min_seconds, args.warmup)
            print(json.dumps(r), flush=True)
            result["cases"].append(r)
    if "host_overlap" in want:
        r = run_host_overlap(torch, lib)
        print(json.dumps(r), flush=True)
        result["host_entry"] = r
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
