"""What the device-resident export costs next to the decode, and what it saves end to end (nafcodec_b200.decode_to_device).

For the bench workload (256 cfg2 archives: 8 distinct 5 Mbp genomes, cycled, as bench.py builds them) and cfg4 (10^6 x 150 bp
FASTQ reads) it prints ONE JSON line with
  - the decode's device time (nafgpu_job_time: CUDA graph of one run, L2 flushed before every run);
  - the kernel time of a flat export and of a 1024 bp rows export (CUDA events, L2 flushed, the launch queued behind a device
    sleep so that the interval holds the kernel and not the host's enqueue), with algorithmic bytes (bytes read + written)
    over that time against the HBM peak bench.py uses;
  - host in -> CUDA tensors (decode_to_device + sequence(), synchronised) against host in -> host out (decode_batch) and
    host out -> .cuda() (what a PyTorch user did before), on the same inputs in memory.
The card's name and power limit are read in the same run.  Usage: python tools/export_probe.py [--out FILE] [--iters K]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

import _cases as K
import bench
import nafcodec_b200 as N
from nafcodec_b200 import _ffi

FLUSH = None


def kernel_ms(fn, iters):
    """Mean device time of fn's work on the current stream, L2 flushed before each launch."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total = 0.0
    for _ in range(iters):
        FLUSH.fill_(7)
        torch.cuda._sleep(2_000_000)                 # ~1 ms: the export is enqueued before e0 runs
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
    return total / iters


def wall_ms(fn, iters):
    fn()
    torch.cuda.synchronize()
    best = []
    for _ in range(iters):
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best.append((time.perf_counter() - t) * 1e3)
    return float(np.median(best))


def rate(nbytes, ms, peak):
    return {"ms": ms, "algorithmic_bytes": int(nbytes), "GBps": nbytes / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak}


def probe(name, datas, fields, iters, peak):
    lib = _ffi.default_library()
    out = {"archives": len(datas), "input_bytes": sum(len(d) for d in datas)}
    recs = N.decode_to_device(datas, **fields)
    res_total = int(recs.offsets[-1])
    out["records"], out["residues"] = recs.n_records, res_total
    ctx = recs._ctx
    out["decode_device_ms"] = ctx.time_runs(iters, flush_l2=True) / iters
    out["flat_sequence_dna5"] = rate(2 * res_total, kernel_ms(lambda: recs.sequence("dna5"), iters), peak)
    out["flat_sequence_ascii"] = rate(2 * res_total, kernel_ms(lambda: recs.sequence(), iters), peak)
    if fields.get("quality"):
        out["flat_quality_phred33"] = rate(2 * res_total, kernel_ms(lambda: recs.quality(), iters), peak)
    lens = recs.lengths
    for label, rows_of in (("rows_1024_windows", lambda: recs.windows(1024)[1]), ("rows_1024_padded", lambda: torch.stack(
            [torch.arange(recs.n_records, device="cuda"), torch.zeros(recs.n_records, dtype=torch.int64, device="cuda")], 1))):
        rows = rows_of()
        starts = rows[:, 1]
        read = int(torch.clamp(lens[rows[:, 0]] - starts, 0, 1024).sum())
        m = rows.shape[0]
        r = rate(read + 16 * m + 1024 * m, kernel_ms(lambda: recs.rows(rows, 1024, table="dna5"), iters), peak)
        r["rows"] = m
        out[label] = r
    recs.close()
    # end to end, inputs in host memory (bytes), outputs where each path leaves them
    host_fields = dict(fields, id=False, comment=False)
    out["e2e_ms"] = {
        "to_cuda_tensor": wall_ms(lambda: (lambda d: (d.sequence(), d.close()))(N.decode_to_device(datas, **fields)), max(3, iters // 4)),
        "to_host": wall_ms(lambda: N.decode_batch(datas, _library=lib, **host_fields), max(3, iters // 4)),
        "to_host_then_cuda": wall_ms(lambda: torch.frombuffer(bytearray(b"".join(r.sequence for r in N.decode_batch(datas, _library=lib, **host_fields))),
                                                              dtype=torch.uint8).cuda(), max(3, iters // 4)),
    }
    out["e2e_sequence_GBps"] = {k: res_total / (v * 1e-3) / 1e9 for k, v in out["e2e_ms"].items()}
    print(f"[{name}] decode {out['decode_device_ms']:.3f} ms; flat export {out['flat_sequence_dna5']['ms']:.3f} ms "
          f"({100 * out['flat_sequence_dna5']['frac_of_hbm_peak']:.1f} % of HBM peak); e2e {out['e2e_ms']}", file=sys.stderr)
    return out


def main():
    global FLUSH
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--cfg4-reads", type=int, default=1_000_000)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak, peak_src = bench.measured_peak()
    FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    uniq = bench.make_workload(8, 5_000_000, 19, 0)
    result = {"probe": "export_probe", "gpu": smi, "hbm_peak_GBps": peak, "peak_source": peak_src,
              "cfg2_batch256": probe("cfg2 x 256", [uniq[i % 8] for i in range(256)], dict(quality=False), args.iters, peak)}
    if args.cfg4_reads:
        result["cfg4"] = probe(f"cfg4 {args.cfg4_reads} reads", [K.cfg4_fastq(args.cfg4_reads)], dict(quality=True), args.iters, peak)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
