"""Batch-wide k-mer counting (ktb_counter_*): step time of one device add into an empty counter, per-stage kernel time,
Gbases/s and algorithmic bytes/s, next to the same table built from the sparse rows (ktb_sparse_vectorise_device) reduced
with torch, and one end-to-end `kmertools ctr` run.  Prints one JSON object per case and writes the whole run to --out.

Bytes of an add (the model): bases + 16 B per valid window per radix pass (one read and one write of a u64 key) + 16 B
per distinct key (the table written).  Share of peak = bytes / time over the measured copy peak (COPY_PEAK_GBS).
Inputs are generated on the GPU by bench.make_workload_torch (the benchmark's seeded workloads); each add reads more
than the 126 MB of L2 except the small-k case's table."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from tools.bench_sparse import COPY_PEAK_GBS, device_intervals, gpu_identity, timed  # noqa: E402

# (label, bench workload, scale, k)
CASES = [
    ("reads150_k21", "reads150_k5", 1.0, 21),
    ("reads150_k31", "reads150_k5", 1.0, 31),
    ("contigs_k21", "contigs_k4", 1.0, 21),
    ("reads10k_k15", "reads10k_k8", 1.0, 15),
    ("reads150_k5", "reads150_k5", 1.0, 5),
]
STAGES = {"keys": ("count_valid_kernel", "count_keys_kernel"),
          "sort": ("count_upsweep_kernel", "count_scatter_kernel"),
          "rle": ("count_rle_",),
          "merge": ("count_merge_",),
          "scan": ("sparse_scan_",)}


def stage_breakdown(iv) -> dict:
    out = {}
    for name, a, b in iv:
        for stage, pats in STAGES.items():
            if any(p in name for p in pats):
                out[stage + "_ms"] = out.get(stage + "_ms", 0.0) + (b - a) / 1e3
    return out


def run_case(torch, case, min_seconds, warmup):
    import bench
    from kmertools_b200 import KmerCounter, _lib
    label, wl, scale, k = case
    dev = torch.device("cuda", 0)
    tb, to = bench.make_workload_torch(bench.WORKLOADS[wl], scale, dev)
    n = to.numel() - 1
    total = int(to[-1])

    def add():
        c = KmerCounter(k)
        c.add_tensors(tb, to)
        return c

    c = add()
    nkeys, nwin = len(c), c.windows
    keys, counts = c.result_tensors()
    c.close()
    ms, steps = timed(torch, lambda: add().close(), min_seconds, warmup)
    stages = stage_breakdown(device_intervals(torch, lambda: add().close()))
    passes = (2 * k + 7) // 8
    nbytes = total + 16 * nwin * passes + 16 * nkeys
    out = {"case": label, "workload": wl, "scale": scale, "k": k, "n": n, "bases": total, "windows": nwin,
           "distinct_keys": nkeys, "radix_passes": passes, "add_ms": ms, "add_steps": steps,
           "gbases_s": total / ms / 1e6, "model_bytes": nbytes, "gb_s": nbytes / ms / 1e6,
           "share_of_copy_peak": nbytes / ms / 1e6 / COPY_PEAK_GBS, "profiled_kernels_ms": stages}

    # the in-repo alternative: sparse rows of the same batch (ktb_sparse_vectorise_device, u32 counts), reduced by code
    # with torch.  The raw entry point, because a torch.sparse_csr_tensor of 4^31 columns overflows its element count.
    def via_sparse():
        row_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        codes = torch.empty(total, dtype=torch.int64, device=dev)
        values = torch.empty(total, dtype=torch.int32, device=dev)
        _lib.check(_lib.load().ktb_sparse_vectorise_device(
            tb.data_ptr(), to.data_ptr(), n, total, k, 1, _lib.NORM_COUNTS, _lib.OUT_U32, row_ptr.data_ptr(),
            codes.data_ptr(), values.data_ptr(), total, None, torch.cuda.current_stream(dev).cuda_stream))
        nnz = int(row_ptr[-1])
        u, inv = torch.unique(codes[:nnz], return_inverse=True)
        s = torch.zeros(len(u), dtype=torch.int64, device=dev)
        s.index_add_(0, inv, values[:nnz].to(torch.int64))
        return u, s
    try:
        u, s = via_sparse()
        out["sparse_reduce_equal"] = bool(torch.equal(u, keys) and torch.equal(s, counts))
        del u, s
        sms, ssteps = timed(torch, via_sparse, min_seconds, warmup)
        out.update(sparse_reduce_ms=sms, sparse_reduce_steps=ssteps, counter_speedup=sms / ms)
    except (RuntimeError, torch.cuda.OutOfMemoryError) as exc:
        out["sparse_reduce_error"] = str(exc).splitlines()[0]
    del tb, to, keys, counts
    torch.cuda.empty_cache()
    return out


def run_cli(tmp: Path, scale: float):
    """`kmertools ctr -k 21` on a FASTQ of the reads150 workload (scale of its 10 M reads): wall time and bytes."""
    import bench
    bases, offsets = bench.make_workload(bench.WORKLOADS["reads150_k5"], scale, bench._NP())
    bases, offsets = np.asarray(bases), np.asarray(offsets)
    fq = tmp / "reads.fq"
    with open(fq, "wb") as f:
        qual = b"I" * 150
        for i in range(len(offsets) - 1):
            s = bases[int(offsets[i]):int(offsets[i + 1])].tobytes()
            f.write(b"@r\n" + s + b"\n+\n" + qual[:len(s)] + b"\n")
    binary = ROOT / "kmertools_b200" / "bin" / "kmertools"
    t0 = time.time()
    r = subprocess.run([str(binary), "ctr", "-i", str(fq), "-o", str(tmp / "out"), "-k", "21"], capture_output=True,
                       text=True, env={**os.environ, "KTB_VERBOSE": "1"})
    wall = time.time() - t0
    out_file = tmp / "out" / "kmers.counts"
    return {"case": "cli_ctr_reads150_k21", "reads": len(offsets) - 1, "bases": int(offsets[-1]),
            "input_bytes": fq.stat().st_size, "wall_s": wall, "bytes_written": out_file.stat().st_size,
            "returncode": r.returncode, "stderr": r.stderr.strip()}


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default="bench_count.json")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES) + ",cli")
    ap.add_argument("--cli-scale", type=float, default=0.2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_count needs a CUDA device")
    result = {"tool": "tools/bench_count.py", **gpu_identity(), "copy_peak_gb_s": COPY_PEAK_GBS,
              "bytes_model": "bases + 16 B per valid window per radix pass + 16 B per distinct key",
              "min_seconds": args.min_seconds, "cases": []}
    want = set(args.cases.split(","))
    for case in CASES:
        if case[0] in want:
            r = run_case(torch, case, args.min_seconds, args.warmup)
            print(json.dumps(r), flush=True)
            result["cases"].append(r)
    if "cli" in want:
        with tempfile.TemporaryDirectory() as d:
            r = run_cli(Path(d), args.cli_scale)
        print(json.dumps(r), flush=True)
        result["cli"] = r
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
