"""Per-read k-mer coverage histograms (ktb_counter_coverage_device): CUDA-event time of one steady-state call, the
directory build of the first call after an add, per-kernel time from one torch.profiler run, windows/s and the table's
size against the 126 MB L2, next to a baseline built from existing primitives in the same process: the sparse rows of
the batch (ktb_sparse_vectorise_device), torch.searchsorted of their codes into the table and scatter_add_ into the bins.
Both give the same u32 rows on every case (checked).  Prints one JSON object per case and writes the run to --out.

Workloads (bench.make_workload_torch, generated on the GPU): the 10 M x 150 bp reads against a table of the same reads
at k = 15 and 21, and the 20 k contigs at k = 15 against a table of 1 M reads of other data, so most keys are absent."""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from tools.bench_sparse import device_intervals, gpu_identity, timed  # noqa: E402

L2_BYTES = 126 * 2 ** 20
BIN_SIZE, BIN_COUNT = 1, 16
# (label, rows workload, table workload, table scale, k)
CASES = [
    ("reads150_k15", "reads150_k5", "reads150_k5", 1.0, 15),
    ("reads150_k21", "reads150_k5", "reads150_k5", 1.0, 21),
    ("contigs_k15", "contigs_k4", "reads150_k5", 0.1, 15),
]


def kernel_ms(iv) -> dict:
    out = {}
    for name, a, b in iv:
        key = next((k for k in ("cov_dir_kernel", "cov_hist_kernel", "cov_write_kernel", "sparse_", "Memset")
                    if k in name), "other")
        out[key + "_ms"] = out.get(key + "_ms", 0.0) + (b - a) / 1e3
    return out


def run_case(torch, case, min_seconds, warmup):
    import bench
    from kmertools_b200 import KmerCounter, _lib
    label, wl, twl, tscale, k = case
    dev = torch.device("cuda", 0)
    tb, to = bench.make_workload_torch(bench.WORKLOADS[wl], 1.0, dev)
    if twl == wl and tscale == 1.0:
        cb, co = tb, to
    else:
        cb, co = bench.make_workload_torch(bench.WORKLOADS[twl], tscale, dev)
    n, total = to.numel() - 1, tb.numel()
    L = _lib.load()

    def fresh():
        c = KmerCounter(k)
        c.add_tensors(cb, co)
        return c

    def call(c, out, norm, dt):
        _lib.check(L.ktb_counter_coverage_device(c._h, tb.data_ptr(), to.data_ptr(), n, total, BIN_SIZE, BIN_COUNT,
                                                 norm, dt, out.data_ptr(), None,
                                                 torch.cuda.current_stream(dev).cuda_stream))

    rows_u32 = torch.empty((n, BIN_COUNT), dtype=torch.int32, device=dev)
    rows_f32 = torch.empty((n, BIN_COUNT), dtype=torch.float32, device=dev)
    c = fresh()
    nkeys = len(c)
    keys, counts = c.result_tensors()
    torch.cuda.synchronize()
    # first call after the add: builds the directory (and waits for it), then enqueues the histogram
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    call(c, rows_f32, _lib.NORM_CLI, _lib.OUT_F32)
    b.record()
    b.synchronize()
    first_ms, first_wall_ms = a.elapsed_time(b), (time.perf_counter() - t0) * 1e3
    steady_f32, s1 = timed(torch, lambda: call(c, rows_f32, _lib.NORM_CLI, _lib.OUT_F32), min_seconds, warmup)
    steady_u32, s2 = timed(torch, lambda: call(c, rows_u32, _lib.NORM_COUNTS, _lib.OUT_U32), min_seconds, warmup)
    kernels = kernel_ms(device_intervals(torch, lambda: call(c, rows_f32, _lib.NORM_CLI, _lib.OUT_F32)))
    c.close()
    c2 = fresh()   # a second table of the same data: the profile of a first call, directory build included
    first_kernels = kernel_ms(device_intervals(torch, lambda: call(c2, rows_f32, _lib.NORM_CLI, _lib.OUT_F32)))
    c2.close()
    dir_bits = min(max(nkeys, 1).bit_length() - 1, 2 * k, 30)
    windows = int(rows_u32.to(torch.int64).sum())
    out = {"case": label, "rows_workload": wl, "table_workload": twl, "table_scale": tscale, "k": k, "n": n,
           "bases": total, "windows": windows, "bin_size": BIN_SIZE, "bin_count": BIN_COUNT,
           "table_keys": nkeys, "table_bytes": 16 * nkeys, "dir_bits": dir_bits, "dir_bytes": 8 * (2 ** dir_bits + 1),
           "table_over_l2": 16 * nkeys / L2_BYTES,
           "first_call_ms": first_ms, "first_call_wall_ms": first_wall_ms,
           "dir_build_kernel_ms": first_kernels.get("cov_dir_kernel_ms", 0.0),
           "call_f32_ms": steady_f32, "call_f32_steps": s1, "call_u32_ms": steady_u32, "call_u32_steps": s2,
           "windows_per_s": windows / steady_f32 * 1e3, "profiled_kernels_ms": kernels,
           "profiled_first_call_kernels_ms": first_kernels}
    # the first call less a steady one: the directory's allocation, its kernel and the wait for it
    out["dir_build_ms"] = first_ms - steady_f32
    out["dir_build_share_of_first_call"] = out["dir_build_ms"] / first_ms

    # the baseline from existing primitives: sparse rows, searchsorted into the table, scatter_add_ into the bins
    def baseline():
        row_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        codes = torch.empty(total, dtype=torch.int64, device=dev)
        values = torch.empty(total, dtype=torch.int32, device=dev)
        _lib.check(L.ktb_sparse_vectorise_device(
            tb.data_ptr(), to.data_ptr(), n, total, k, 1, _lib.NORM_COUNTS, _lib.OUT_U32, row_ptr.data_ptr(),
            codes.data_ptr(), values.data_ptr(), total, None, torch.cuda.current_stream(dev).cuda_stream))
        nnz = int(row_ptr[-1])
        codes, values = codes[:nnz], values[:nnz]
        at = torch.searchsorted(keys, codes).clamp_(max=max(nkeys - 1, 0))
        absent = keys[at] != codes
        ab = counts[at]
        del at
        ab.masked_fill_(absent, 0).floor_divide_(BIN_SIZE).clamp_(max=BIN_COUNT - 1)
        del absent
        seq = torch.repeat_interleave(torch.arange(n, device=dev), row_ptr[1:] - row_ptr[:-1], output_size=nnz)
        seq.mul_(BIN_COUNT).add_(ab)
        del ab
        rows = torch.zeros(n * BIN_COUNT, dtype=torch.int64, device=dev)
        rows.scatter_add_(0, seq, values.to(torch.int64))
        return rows
    try:
        want = baseline()
        out["baseline_equal"] = bool(torch.equal(want, rows_u32.to(torch.int64).view(-1)))
        del want
        bms, bsteps = timed(torch, baseline, min_seconds, warmup)
        out.update(baseline_ms=bms, baseline_steps=bsteps, speedup_over_baseline=bms / steady_u32,
                   profiled_baseline_ms=kernel_ms(device_intervals(torch, baseline)))
    except (RuntimeError, torch.cuda.OutOfMemoryError) as exc:
        out["baseline_error"] = str(exc).splitlines()[0]
    del tb, to, cb, co, keys, counts, rows_u32, rows_f32
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default="profiles/cov_bench.json")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_cov needs a CUDA device")
    result = {"tool": "tools/bench_cov.py", **gpu_identity(), "l2_bytes": L2_BYTES, "min_seconds": args.min_seconds,
              "cases": []}
    want = set(args.cases.split(","))
    for case in CASES:
        if case[0] in want:
            r = run_case(torch, case, args.min_seconds, args.warmup)
            print(json.dumps(r), flush=True)
            result["cases"].append(r)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
