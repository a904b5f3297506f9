#!/usr/bin/env python
"""bench.py -- measures the nafcodec hot path (zstd NAF sections -> per-record ASCII) on B200.

Contract (one JSON line on stdout, rank 0):
  metric  : decoded GB/s of ASCII out (BASELINE.json), whole job over all GPUs
  value   : device-resident throughput: compressed sections + block descriptors already in HBM when the timed region
            starts; CUDA events on the stream the kernels are launched on; max over ranks
  e2e     : same metric through the public C-ABI call nafgpu_decode_batch with HOST buffers (pinned), H2D and D2H inside
            the timed region
  roofline: dominant kernel's algorithmic bytes / its measured duration vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline: the CPU oracle (C restatement of the reference decoder on libzstd; the Rust reference cannot be built in
            this image) timed on a bounded sample of the same workload, 1 thread (the reference is single-threaded)
A "step" = one decode of a batch of `--batch` independent cfg2 archives (synthetic 5 Mbp bacterial genome, single
record, 4-bit sequence + soft-mask runs, zstd level 19) per GPU.  Archives are partitioned across GPUs with no
collective (nothing reduces): weak scaling.
`--impl reference` times the reference's CPU path instead (oracle port, all host cores, one archive per core).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "decoded_ascii_GBps"
UNIT = "GB/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on stdout.  Keep a private copy
# of the real stdout for that line and point fd 1 at stderr for everything else.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


# ------------------------------------------------------------------------------------------------------------------
# workload: cfg2 archives, generated with the oracle's restatement of the reference encoder (+ mask section)
def make_archive(seed, n_res, level):
    import _cases as K
    return K.cached(f"cfg2_s{seed}_n{n_res}_l{level}.naf", lambda: K.genome(seed, n_res, level=level, mask=True, records=1))[0]


def make_workload(unique, n_res, level, rank):
    import _oracle as O
    O.lib()
    seeds = [1000 + rank * unique + i for i in range(unique)]
    with ThreadPoolExecutor(max_workers=min(unique, os.cpu_count() or 1)) as ex:     # ctypes releases the GIL
        return list(ex.map(lambda s: make_archive(s, n_res, level), seeds))


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks/throttle reasons for one GPU while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.proc = p
        for line in p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])
            if self.stop_flag.is_set():
                break
        p.kill()

    def summary(self):
        self.stop_flag.set()
        time.sleep(0.15)
        try:
            self.proc.kill()
        except Exception:
            pass
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------
def cpu_decode_all(archives, threads, want_quality=True, want_mask=True):
    """Reference CPU path (oracle port): one archive per core at a time on a NATIVE thread pool inside libnaforacle.so (no
    interpreter between the archives, buffers stay on the threads' malloc arenas).  Returns (seconds, ascii bytes)."""
    import _oracle as O
    return O.time_decode_many(archives, threads, quality=want_quality, mask=want_mask)


def run_reference(args, rank, world):
    if rank != 0:
        return
    import _oracle as O
    cores = os.cpu_count() or 1
    uniq = make_workload(args.unique, args.residues, args.level, 0)
    sample_n = args.batch                     # the same batch as the device arm (256 cfg2 archives: ~3 s of CPU work per step on 16 cores)
    archives = [uniq[i % len(uniq)] for i in range(sample_n)]
    for _ in range(args.warmup):
        cpu_decode_all(archives[:cores], cores)
    total_t, total_b = 0.0, 0
    for _ in range(args.steps):
        t, b = cpu_decode_all(archives, cores)
        total_t += t
        total_b += b
    val = total_b / total_t / 1e9
    # per-core rate at 1 thread and at all of them (a CPU arm that loses its per-core rate at high thread counts flatters the GPU)
    t1, b1 = cpu_decode_all(archives[:8], 1)
    per_core = {"1_thread_GBps": b1 / t1 / 1e9, f"{cores}_threads_GBps_per_core": val / cores}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_t / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": workload_config(args, sample_n),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "per_core": per_core,
                             "sample": f"{sample_n} cfg2 archives per step, one archive per core at a time, {cores} native threads; oracle/naf_oracle.c on libzstd {O.lib().nafo_zstd_version().decode()} (the Rust reference cannot be built in this image: no cargo/rustc)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(args, batch):
    return {"workload": f"cfg2: synthetic {args.residues / 1e6:g} Mbp bacterial genome, single-record DNA, 4-bit sequence + soft-mask runs, zstd level {args.level}; "
                        f"decode sequence+mask+ids+comments+lengths",
            "archives_per_gpu_per_step": batch, "unique_archives_per_gpu": args.unique, "residues_per_archive": args.residues,
            "zstd_level": args.level, "parallelism": f"archives partitioned over {args.gpus} GPU(s), no collective",
            "l2": "batch working set (compressed + packed + ASCII) exceeds the 126 MB L2; device-resident timing also overwrites a 256 MB buffer before every timed iteration"}


DUMP_SEED = 20261020
DUMP_SEQUENCE_SAMPLES = 8 << 20            # float32: 32 MiB, the largest of the files


def dump_outputs(out_dir, results):
    """What a caller of the timed decode receives for the batch, as exact float arrays: n_records per archive, every record
    length (float64), the ids and comments blobs (NUL-terminated, archives concatenated) and the sequence bytes of each
    archive, whole if it fits its share of DUMP_SEQUENCE_SAMPLES, else at a fixed seeded sample of positions (the batch is
    1.28 GB of ASCII at the default sizes; float32)."""
    import numpy as np

    def view(ptr, n, ctype):
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(n,)) if ptr and n else np.zeros(0, np.dtype(ctype))

    n_arc = len(results)
    per_archive = DUMP_SEQUENCE_SAMPLES // n_arc
    out = {"n_records": [], "lengths": [], "ids": [], "comments": [], "sequence_sample": []}
    for i, r in enumerate(results):
        assert r.status == 0, (i, r.status)
        out["n_records"].append(np.array([r.n_records], np.float64))
        out["lengths"].append(view(r.lengths, r.n_lengths, C.c_uint64).astype(np.float64))
        for name, blob, offsets, n in (("ids", r.ids, r.id_offsets, r.n_ids), ("comments", r.comments, r.comment_offsets, r.n_comments)):
            size = int(view(offsets, n + 1, C.c_uint64)[-1]) if blob else 0
            out[name].append(view(blob, size, C.c_uint8).astype(np.float32))
        seq = view(r.sequence, r.total_residues, C.c_uint8)
        if len(seq) > per_archive:
            seq = seq[np.sort(np.random.default_rng([DUMP_SEED, i]).integers(0, len(seq), size=per_archive))]
        out["sequence_sample"].append(seq.astype(np.float32))
    os.makedirs(out_dir, exist_ok=True)
    for name, parts in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.concatenate(parts))
    log(f"[dump] {len(out)} arrays of the last timed step written to {out_dir}")


# ------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs at their stated sizes, each: parity gate vs the oracle, host prepare, device time, roofline, e2e
def pin(lib, blobs):
    """Pinned host copies + parsed archive structs (the e2e legs copy from pinned memory)."""
    from nafcodec_b200 import _ffi
    out, keep = [], []
    for a in blobs:
        p = lib.dll.nafgpu_host_alloc(len(a))
        C.memmove(p, a, len(a))
        keep.append(p)
        arc = _ffi.Archive()
        rc = lib.dll.nafgpu_parse_archive(p, len(a), C.byref(arc))
        assert rc == 0, rc
        out.append(arc)
    return out, keep


def measure_config(ctx, lib, name, blobs, want, peak, fields, note, iters=10, parity_sample=None):
    """One job = all `blobs` decoded together.  Returns the dict that goes under configs[name] in the bench line."""
    import _oracle as O
    from _harness import assert_same_as_oracle
    from nafcodec_b200 import _ffi
    archives, keep = pin(lib, blobs)
    n = len(archives)
    arr = (_ffi.Archive * n)(*archives)
    res = (_ffi.Result * n)()
    # parity gate: device == oracle, every field, on every archive (or on a stated sample of a big collection)
    idx = list(range(n)) if parity_sample is None else parity_sample
    t0 = time.perf_counter()
    got = ctx.decode(archives, want)
    t_first = time.perf_counter() - t0
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=min(len(idx), os.cpu_count() or 1)) as ex:
        wants = list(ex.map(lambda i: O.decode(blobs[i], **fields), idx))
    t_cpu = time.perf_counter() - t0
    for i, w in zip(idx, wants):
        assert_same_as_oracle(got[i], w, f"{name} archive {i}")
    del got, wants
    # host prepare: frame/block header walk + descriptor build + H2D enqueue (buffers exist after the first call)
    preps = []
    for _ in range(3):
        t0 = time.perf_counter()
        ctx.prepare(archives, want)
        preps.append(time.perf_counter() - t0)
        ctx.sync()
    st = ctx.stats()
    ctx.time_runs(2, True)
    ms = ctx.time_runs(iters, True) / iters
    stages = {nm: round(v, 4) for nm, v in ctx.profile_stages() if v >= 0.0005}
    ctx.fetch_raw()
    st2 = ctx.stats()
    # end to end through the C ABI: pinned host buffers in, pinned host buffers out, one synchronous call
    e2es = []
    for _ in range(3):
        t0 = time.perf_counter()
        rc = lib.dll.nafgpu_decode_batch(ctx._ctx, arr, n, want, res)
        e2es.append(time.perf_counter() - t0)
        assert rc == 0, rc
    # the same call when the caller bounds its host memory (DecoderBuilder::buffer_size): decode into HBM, records of archive 0
    # fetched in windows of 1 MiB of decoded data (nafgpu_job_fetch_window); time to the first window, and to the last one
    win = _ffi.Result()
    firsts, alls = [], []
    n_windows = 0
    for _ in range(3):
        t0 = time.perf_counter()
        rc = lib.dll.nafgpu_job_prepare(ctx._ctx, arr, n, want) or lib.dll.nafgpu_job_run(ctx._ctx)
        assert rc == 0, rc
        i, n_windows, n_rec = 0, 0, int(arr[0].header.number_of_sequences)
        while i < n_rec:
            rc = lib.dll.nafgpu_job_fetch_window(ctx._ctx, 0, i, n_rec - i, 1 << 20, C.byref(win))
            assert rc == 0 and win.n_records > 0, (rc, i)
            if i == 0:
                firsts.append(time.perf_counter() - t0)
            i += int(win.n_records)
            n_windows += 1
        alls.append(time.perf_counter() - t0)
    out_bytes = int(st.ascii_bytes + st.quality_bytes + st.id_bytes + st.comment_bytes)
    e2e_s = sorted(e2es)[1]
    prep_ms = sorted(preps)[1] * 1e3
    for p in keep:
        lib.dll.nafgpu_host_free(p)
    return {"workload": note, "archives": n, "parity": f"bit-exact vs oracle on {len(idx)} archive(s), all requested fields",
            "zstd_blocks": int(st.n_blocks), "sequences": int(st.n_sequences), "kernel_launches": int(st2.kernel_launches),
            "compressed_bytes": int(st.compressed_bytes), "ascii_bytes": int(st.ascii_bytes), "output_bytes": out_bytes,
            "algorithmic_bytes": int(st.algorithmic_bytes),
            "device_ms": ms, "host_prepare_ms": prep_ms, "device_plus_prepare_ms": ms + prep_ms,
            "ascii_GBps": int(st.ascii_bytes) / (ms * 1e-3) / 1e9, "output_GBps": out_bytes / (ms * 1e-3) / 1e9,
            "path_algorithmic_GBps": int(st.algorithmic_bytes) / (ms * 1e-3) / 1e9,
            "frac_of_hbm_peak": int(st.algorithmic_bytes) / (ms * 1e-3) / 1e9 / peak,
            "e2e": {"ms": e2e_s * 1e3, "output_GBps": out_bytes / e2e_s / 1e9, "h2d_bytes": int(st.h2d_bytes), "d2h_bytes": int(st.d2h_bytes),
                    "first_call_ms": t_first * 1e3,
                    "windowed": {"window_bytes": 1 << 20, "archive": 0, "windows": n_windows, "first_window_ms": sorted(firsts)[1] * 1e3,
                                 "all_windows_ms": sorted(alls)[1] * 1e3}},
            "lz_rounds": int(st2.lz_rounds), "lz_handover_round": int(st2.lz_handover), "lz_in_order_kernel": int(st2.lz_flow), "stage_ms_serial": stages,
            "cpu_oracle": {"ms": t_cpu * 1e3, "threads": min(len(idx), os.cpu_count() or 1), "archives": len(idx)}}


def run_configs(args, ctx, lib, peak, uniq_cfg2):
    """configs[0..4] of BASELINE.json at their stated sizes (cfg2 x 256 is the headline workload itself)."""
    import _cases as K
    import _oracle as O
    from nafcodec_b200 import _ffi
    out = {}
    ALL = dict(id=True, comment=True, sequence=True, quality=True, mask=True)
    want = _ffi.WANT_ALL

    def guarded(name, fn):
        t0 = time.perf_counter()
        try:
            out[name] = fn()
            out[name]["wall_s"] = round(time.perf_counter() - t0, 1)
            log(f"[configs] {name}: device {out[name]['device_ms']:.3f} ms, prepare {out[name]['host_prepare_ms']:.2f} ms, "
                f"{out[name]['ascii_GBps']:.1f} GB/s ASCII, {100 * out[name]['frac_of_hbm_peak']:.2f} % of HBM peak, e2e {out[name]['e2e']['ms']:.2f} ms")
        except AssertionError:
            raise                                        # a parity failure must fail the bench
        except Exception as e:                           # (generation / memory trouble: say so instead of dropping the line)
            out[name] = {"error": f"{type(e).__name__}: {e}"}

    golden = os.path.join(ROOT, "tests", "golden", "NZ_AAEN01000029.naf")
    guarded("cfg1_fixture", lambda: measure_config(ctx, lib, "cfg1", [open(golden, "rb").read()], want, peak, ALL,
                                                   "cfg1: data/NZ_AAEN01000029.naf (30 records, 5.49 Mbp), all fields", iters=20))
    guarded("cfg2_single", lambda: measure_config(ctx, lib, "cfg2", [uniq_cfg2[0]], want, peak, ALL,
                                                  f"cfg2: ONE synthetic {args.residues / 1e6:g} Mbp genome archive alone (latency-bound: the working set sits in L2)", iters=20))
    if args.cfg3_residues > 0:
        def cfg3():
            nm = f"cfg3_n{args.cfg3_residues}_s3_l19.naf"
            data, how = K.cached(nm, lambda: K.cfg3_chromosome(args.cfg3_residues, workers=0))
            r = measure_config(ctx, lib, "cfg3", [data], want, peak, ALL,
                               f"cfg3: synthetic {args.cfg3_residues / 1e6:g} Mbp chromosome, ONE record / one zstd frame per section, level 19 (8 MiB window), "
                               f"N telomeres + centromere + 20 gaps, ~50 % soft-masked (mean run 300); archive {how}", iters=5)
            return r
        guarded("cfg3_250Mbp" if args.cfg3_residues == 250_000_000 else f"cfg3_{args.cfg3_residues // 1_000_000}Mbp", cfg3)
    if args.cfg4_reads > 0:
        nm = f"cfg4_{args.cfg4_reads // 1000}k" if args.cfg4_reads < 1_000_000 else f"cfg4_{args.cfg4_reads // 1_000_000}M"
        data4 = K.cfg4_fastq(args.cfg4_reads)
        note4 = (f"cfg4: {args.cfg4_reads} x 150 bp FASTQ reads, ids + quality + mask, reference encoder framing (zstd flush per record: one tiny block "
                 f"per read and stream), level 0 = the reference default (level 19 with 2e7 flushes is impractical to generate)")
        guarded(nm + "_all_fields", lambda: measure_config(ctx, lib, "cfg4", [data4], want, peak, ALL, note4 + "; all fields", iters=3))
        guarded(nm + "_no_quality", lambda: measure_config(ctx, lib, "cfg4-q", [data4], want & ~_ffi.WANT_QUALITY, peak,
                                                           dict(ALL, quality=False), note4 + "; .quality(false)", iters=3))
        del data4
    if args.cfg5_archives > 0:
        def cfg5():
            t0 = time.perf_counter()
            with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
                blobs = list(ex.map(lambda i: K.cached(f"cfg5_i{i}_l19.naf", lambda: K.cfg5_member(i))[0], range(args.cfg5_archives)))
            gen_s = time.perf_counter() - t0
            r = measure_config(ctx, lib, "cfg5", blobs, want, peak, ALL,
                               f"cfg5: RefSeq-collection shape, {args.cfg5_archives} UNIQUE archives in one job (of the 20 000 / 8 GPUs = 2500 per GPU), N uniform 2-6 Mbp, "
                               f"1 chromosome + 0-3 plasmid records, level 19; generated in {gen_s:.0f} s on {os.cpu_count()} host threads", iters=5)
            return r
        guarded(f"cfg5_mix_{args.cfg5_archives}", cfg5)
    return out


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="archives per GPU per step (the collection shape: cfg5 is 2500 per GPU; 64 gives 259 GB/s, 256 307, 1024 325)")
    ap.add_argument("--unique", type=int, default=8, help="distinct generated archives per GPU (cycled to fill the batch)")
    ap.add_argument("--residues", type=int, default=5_000_000)
    ap.add_argument("--level", type=int, default=19)
    ap.add_argument("--lanes", type=int, default=4, help="contexts (streams) used by the end-to-end leg")
    ap.add_argument("--cfg3-residues", type=int, default=250_000_000, help="configs[2]: one chromosome-scale archive (0 = skip)")
    ap.add_argument("--cfg4-reads", type=int, default=1_000_000, help="configs[3]: FASTQ reads (BASELINE says 10 M: 450 MB archive, ~2 min to generate; 0 = skip)")
    ap.add_argument("--cfg5-archives", type=int, default=512, help="configs[4]: unique 2-6 Mbp archives in one job (0 = skip)")
    ap.add_argument("--no-configs", action="store_true", help="only the headline workload (cfg2 x batch)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step decoded (rank 0) to DIR/<name>.npy, "
                                                          "so that two builds can be compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import nafcodec_b200 as N
    from nafcodec_b200 import _ffi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: nafcodec_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    lib = _ffi.default_library()
    ctx = N.Context(local, lib)
    uniq = make_workload(args.unique, args.residues, args.level, rank)
    # pinned host copies of the archives: the e2e leg copies from pinned memory
    pinned = []
    for a in uniq:
        p = lib.dll.nafgpu_host_alloc(len(a))
        C.memmove(p, a, len(a))
        pinned.append((p, len(a)))
    archives = []
    for i in range(args.batch):
        p, n = pinned[i % len(pinned)]
        arc = _ffi.Archive()
        rc = lib.dll.nafgpu_parse_archive(p, n, C.byref(arc))
        assert rc == 0, rc
        archives.append(arc)
    want = _ffi.WANT_ALL

    # ---- parity gate before any timing (BASELINE.md 4): device == oracle on the workload's archives ------------------
    import _oracle as O
    from _harness import assert_same_as_oracle
    got = ctx.decode(archives[:len(uniq)], want)
    for i, a in enumerate(uniq):
        assert_same_as_oracle(got[i], O.decode(a), f"bench archive {i}")
    log(f"[rank {rank}] parity gate ok on {len(uniq)} archives")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput ---------------------------------------------------------------------------------
    ctx.prepare(archives, want)
    ctx.sync()
    st = ctx.stats()
    ctx.time_runs(args.warmup, True)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    dev_ms = ctx.time_runs(args.steps, True)
    barrier()
    dev_ms = max_over_ranks(dev_ms)
    res = ctx.fetch_raw()                  # (outside the timed region) the last run's results and its LZ round statistics
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)
    st = ctx.stats()                       # kernel_launches is filled by the runs
    lz_rounds = int(st.lz_rounds)
    ascii_bytes = st.ascii_bytes
    value = world * ascii_bytes * args.steps / (dev_ms * 1e-3) / 1e9

    # ---- per-stage times (events on the launch stream) for the roofline of the dominant kernel -----------------------
    stage_acc = None
    reps = 5
    for _ in range(reps):
        s = ctx.profile_stages()
        stage_acc = [x[1] for x in s] if stage_acc is None else [a + x[1] for a, x in zip(stage_acc, s)]
    stage_names = [x[0] for x in s]
    stage_ms = [a / reps for a in stage_acc]
    kern_ms = dict(zip(stage_names, stage_ms)).get("huf_big_kernel", 0.0)     # the dominant kernel alone (own event pair)
    stage_names, stage_ms = stage_names[:-1], stage_ms[:-1]
    dom = max(range(len(stage_ms)), key=lambda i: stage_ms[i])
    lits = st.section_bytes                # every regenerated section byte is produced once by the zstd stage
    kernel_bytes = {                       # algorithmic bytes per launch of each stage (DESIGN.md "Kernels")
        "memset+huf_decode": st.compressed_bytes + lits,
        "unpack": lits + st.ascii_bytes,
        "decode_sequences": st.compressed_bytes,
        "lz_literals": 2 * lits, "lz_first": 2 * lits, "lz_resolve": 2 * lits,
    }
    dom_name = stage_names[dom]
    kernel_of = {"memset+huf_decode": "k_huf_decode_block", "decode_sequences": "k_decode_sequences", "unpack": "k_unpack",
                 "lz_resolve": "k_lz_resolve", "lz_first": "k_lz_first", "lz_literals": "k_lz_literals", "build_tables": "k_build_tables<0>"}
    dom_bytes = kernel_bytes.get(dom_name, st.algorithmic_bytes)
    peak, peak_src = measured_peak()
    # DRAM traffic of the dominant kernel per launch, from the committed `ncu --set full` capture (profiles/r2_traffic.json)
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        ent = tj.get(kernel_of.get(dom_name, dom_name))
        if ent and ent.get("archives") == args.batch:
            traffic, traffic_src = ent["dram_bytes_per_launch"], ent["source"]
    dom_ms = kern_ms if (dom_name == "memset+huf_decode" and kern_ms > 0) else stage_ms[dom]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    path_gbs = st.algorithmic_bytes * args.steps / (dev_ms * 1e-3) / 1e9

    # ---- end to end through the C ABI: pinned host in, pinned host out ------------------------------------------------
    # The batch is split over `--lanes` contexts driven from host threads (the public Pipeline API), so that H2D, kernels
    # and D2H of different sub-batches overlap; every byte of input and output still crosses PCIe inside the timed region.
    pipe = N.Pipeline(local, args.lanes, lib)
    seen = [0]

    def consume(i, r):
        seen[0] += int(r.total_residues)          # touch the result struct: the pinned output is ready here

    def consume_s(bi, i, r):
        seen[0] += int(r.total_residues)

    # (1) one synchronous call per step: Pipeline.decode waits for every lane before the next step starts
    for _ in range(args.warmup):
        pipe.decode(archives, want, consume)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pipe.decode(archives, want, consume)
    torch.cuda.synchronize()
    sync_s = time.perf_counter() - t0
    barrier()
    sync_s = max_over_ranks(sync_s)
    # (2) the K steps submitted as one stream of batches (Pipeline.decode_stream): the lanes pull sub-batches with no barrier
    # between steps, so one step's D2H overlaps the next step's header walk, H2D and kernels.  Same bytes over PCIe per step.
    pipe.decode_stream([archives] * args.warmup, want, consume_s)
    barrier()
    t0 = time.perf_counter()
    n_done = pipe.decode_stream([archives] * args.steps, want, consume_s)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_s = max_over_ranks(e2e_s)
    assert n_done == args.steps * len(archives)
    lane_stats = pipe.stats()
    h2d_step = sum(int(s.h2d_bytes) for s in lane_stats)
    d2h_step = sum(int(s.d2h_bytes) for s in lane_stats)
    assert seen[0] == 2 * (args.steps + args.warmup) * ascii_bytes, (seen[0], ascii_bytes)
    e2e_val = world * ascii_bytes * args.steps / e2e_s / 1e9
    clocks = sampler.summary()

    # ---- what the host <-> device link gives for the SAME bytes with the same concurrency (every rank at the same time): the
    # ceiling of the end-to-end number.  Pure copies, no kernels: `lanes` streams, each H2D then D2H of its share per step.
    ceil_bufs = []
    for _ in range(args.lanes):
        hi = torch.empty(max(h2d_step // args.lanes, 1), dtype=torch.uint8, pin_memory=True)
        ho = torch.empty(max(d2h_step // args.lanes, 1), dtype=torch.uint8, pin_memory=True)
        ceil_bufs.append((hi, ho, torch.empty_like(hi, device="cuda"), torch.empty_like(ho, device="cuda"), torch.cuda.Stream()))

    def copy_steps(k):
        for _ in range(k):
            for hi, ho, di, do, stream in ceil_bufs:
                with torch.cuda.stream(stream):
                    di.copy_(hi, non_blocking=True)
                    ho.copy_(do, non_blocking=True)
        torch.cuda.synchronize()

    copy_steps(args.warmup)
    barrier()
    t0 = time.perf_counter()
    copy_steps(args.steps)
    ceil_s = time.perf_counter() - t0
    barrier()
    ceil_s = max_over_ranks(ceil_s)
    ceil_val = world * ascii_bytes * args.steps / ceil_s / 1e9
    del ceil_bufs

    # ---- FASTA text of the same batch, formatted on the device (SURVEY 8f rank 1; reported beside the metric, not part of it) ----
    text = None
    if rank == 0:
        n_arc = len(archives)
        arr = (_ffi.Archive * n_arc)(*archives)
        texts = (_ffi.Text * n_arc)()
        tms = []
        for _ in range(5):
            rc = lib.dll.nafgpu_format_batch(ctx._ctx, arr, n_arc, want, _ffi.TEXT_FASTA, _ffi.LINE_LENGTH_FROM_HEADER, texts)
            assert rc == 0, rc
            tms.append(float(ctx.stats().text_kernel_ms))
        ts = ctx.stats()
        tmed = sorted(tms)[len(tms) // 2]
        talg = int(ts.text_bytes) + int(ts.ascii_bytes) + int(ts.id_bytes) + int(ts.comment_bytes)
        text = {"format": "fasta", "text_bytes": int(ts.text_bytes), "kernels": ["k_text_layout", "k_text_write"], "device_ms": tmed,
                "text_GBps": int(ts.text_bytes) / (tmed * 1e-3) / 1e9, "algorithmic_bytes": talg,
                "frac_of_hbm_peak": talg / (tmed * 1e-3) / 1e9 / peak}

    # ---- single archive latency (cfg2 as one archive) ------------------------------------------------------------------
    single = None
    if rank == 0:
        ctx.prepare(archives[:1], want)
        ctx.sync()
        s1 = ctx.stats()
        ctx.time_runs(3, True)
        ms1 = ctx.time_runs(20, True) / 20
        s1 = ctx.stats()
        st1 = {nm: round(ms, 4) for nm, ms in ctx.profile_stages()}       # serial: the two branches do not overlap here
        single = {"device_us": ms1 * 1e3, "ascii_GBps": s1.ascii_bytes / (ms1 * 1e-3) / 1e9, "kernel_launches": s1.kernel_launches, "stage_ms_serial": st1,
                  "algorithmic_bytes": s1.algorithmic_bytes, "frac_of_hbm_peak": s1.algorithmic_bytes / (ms1 * 1e-3) / 1e9 / peak}

    # ---- every BASELINE.json config at its stated size (N=1 only: each is a single-GPU job) -------------------------------
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        configs = run_configs(args, ctx, lib, peak, uniq)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample, 1 thread ------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1:
        k = 0
        t_cpu, b_cpu = 0.0, 0
        while t_cpu < 10.0 and k < 400:
            t, b = O.time_decode(uniq[k % len(uniq)], quality=True, mask=True, iters=1)
            t_cpu += t
            b_cpu += b
            k += 1
        cpu = {"value": b_cpu / t_cpu / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"{k} single-archive decodes (~10 s) of the same cfg2 archives, 1 thread; oracle/naf_oracle.c on libzstd "
                         f"{O.lib().nafo_zstd_version().decode()} (Rust reference not buildable here: no cargo/rustc)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": workload_config(args, args.batch),
                "compressed_in_GBps": world * st.compressed_bytes * args.steps / (dev_ms * 1e-3) / 1e9,
                "path_algorithmic_GBps": path_gbs, "path_frac_of_hbm_peak": path_gbs / peak,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step, "lanes": args.lanes, "mode": "K steps streamed through Pipeline.decode_stream (no barrier between steps)",
                        "per_step_sync": {"value": world * ascii_bytes * args.steps / sync_s / 1e9, "ms_per_step": sync_s / args.steps * 1e3},
                        "ms_per_step": e2e_s / args.steps * 1e3,
                        "ceiling": {"value": ceil_val, "unit": UNIT, "ms_per_step": ceil_s / args.steps * 1e3,
                                    "what": f"pure copies of the same {h2d_step} B H2D + {d2h_step} B D2H per step and GPU over {args.lanes} streams from pinned memory, "
                                            f"all {world} rank(s) at once, expressed in the metric's unit (ASCII bytes / time)"},
                        "frac_of_ceiling": e2e_val / ceil_val},
                "gpu_launches": int(st.kernel_launches) * args.steps,
                "roofline": {"bound": "hbm", "kernel": kernel_of.get(dom_name, dom_name), "stage": dom_name, "traffic_source": traffic_src, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "peak_source": peak_src, "kernel_ms": dom_ms, "algorithmic_bytes_per_launch": int(dom_bytes),
                             "stage_ms": {nm: round(ms, 4) for nm, ms in zip(stage_names, stage_ms)}},
                "cpu_baseline": cpu, "clocks": clocks, "single_archive": single, "text_formatter": text, "configs": configs,
                "job": {"archives": int(st.n_archives), "frames": int(st.n_frames), "zstd_blocks": int(st.n_blocks), "sequences": int(st.n_sequences), "lz_rounds": lz_rounds,
                        "compressed_bytes": int(st.compressed_bytes), "ascii_bytes": int(st.ascii_bytes), "algorithmic_bytes": int(st.algorithmic_bytes)}}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
