"""What the lanes of stream_to_device buy over decoding a collection sub-batch by sub-batch (nafcodec_b200.stream_to_device).

A collection of the cfg5 shape (unique 2-6 Mbp level-19 archives of tests/_cases.cfg5_member, from the per-user archive
cache, cycled to --archives), inputs in host memory as bytes, cut into the same sub-batches by the rule of stream_to_device.
These arms run alternately, --rounds times each, every one ending in a device synchronise:
  serial      decode_to_device per sub-batch, one after the other, one flat export of the sequence each
  lanes_L     stream_to_device at lanes L (1, 2, 3) with the same sub-batches and the same export
  h2d         cudaMemcpyAsync (torch copy_ from pinned memory) of the same compressed bytes, archive by archive: the input-side
              ceiling, since every arm has to move these bytes to the device
For each arm it reports the median wall time, GB/s of ASCII produced in HBM and the fraction of the h2d ceiling (h2d time over
the arm's time), the peak of torch.cuda.max_memory_allocated, and the peak of device memory outside torch's allocator above
what the process held before the arm (the lanes' arenas; device-wide, as cudaMemGetInfo sees it).  The card's name and power
limit are read in the same run.  Before the timed rounds, every arm's output is checked against the serial arm's.

    python tools/stream_probe.py --out FILE                     # a B200: 4096 archives, 256 MB sub-batches
    python tools/stream_probe.py --emul --archives 12 --unique 4 --batch-bytes 60000    # the emulator library, tiny archives
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch

import _cases as K
import nafcodec_b200 as N


def cuts_of(sizes, batch_bytes, max_archives=65535):
    """[(lo, hi)] of the sub-batches stream_to_device cuts (its documented rule)."""
    out, lo, size = [], 0, 0
    for i, s in enumerate(sizes):
        if i > lo and (size + s > batch_bytes or i - lo == max_archives):
            out.append((lo, i))
            lo, size = i, 0
        size += s
    if sizes:
        out.append((lo, len(sizes)))
    return out


class Arm:
    """Runs one arm and tracks its memory: torch's peak allocation and device memory outside torch above the start."""

    def __init__(self, cuda):
        self.cuda = cuda

    def __enter__(self):
        if self.cuda:
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            self.base = self._outside()
        self.peak_outside = 0
        self.t0 = time.perf_counter()
        return self

    def _outside(self):
        free, total = torch.cuda.mem_get_info()
        return total - free - torch.cuda.memory_reserved()

    def sample(self):
        if self.cuda:
            self.peak_outside = max(self.peak_outside, self._outside() - self.base)

    def __exit__(self, *exc):
        if self.cuda:
            torch.cuda.synchronize()
        self.seconds = time.perf_counter() - self.t0
        self.peak_torch = torch.cuda.max_memory_allocated() if self.cuda else None
        return False


def drop_pool():
    """Closes the pooled contexts decode_to_device keeps, so that every arm starts from the same device memory."""
    with N.device._pool_lock:
        for idle in N.device._pool.values():
            for ctx in idle:
                ctx.close()
        N.device._pool.clear()


def digest(x):
    """A position-weighted sum of an export (a check that two arms wrote the same bytes, outside the timed rounds)."""
    w = torch.arange(x.numel(), device=x.device, dtype=torch.int64) % 251 + 1
    return int((x.to(torch.int64) * w).sum())


def run_serial(datas, cuts, kw, cuda, check=None):
    out = []
    with Arm(cuda) as arm:
        for lo, hi in cuts:
            recs = N.decode_to_device(datas[lo:hi], quality=False, **kw)
            x = recs.sequence()
            arm.sample()
            out.append(digest(x) if check else x.numel())
            recs.close()
            del x
    return arm, out


def run_stream(datas, batch_bytes, lanes, kw, cuda, check=None):
    out = []
    with Arm(cuda) as arm:
        for recs in N.stream_to_device(datas, batch_bytes=batch_bytes, lanes=lanes, quality=False, **kw):
            x = recs.sequence()
            arm.sample()
            out.append(digest(x) if check else x.numel())
            recs.close()
            del x
    return arm, out


def run_h2d(pinned, order, cuts, sizes):
    dst = torch.empty(max(sum(sizes[lo:hi]) for lo, hi in cuts), dtype=torch.uint8, device="cuda")
    with Arm(True) as arm:
        for lo, hi in cuts:
            at = 0
            for i in range(lo, hi):
                dst[at:at + sizes[i]].copy_(pinned[order[i]], non_blocking=True)
                at += sizes[i]
    return arm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--archives", type=int, default=4096)
    ap.add_argument("--unique", type=int, default=64)
    ap.add_argument("--batch-bytes", type=int, default=256 << 20)
    ap.add_argument("--lanes", default="1,2,3")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--emul", action="store_true", help="the CPU emulator library and tiny archives (a dry run without a GPU)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lanes_list = [int(x) for x in args.lanes.split(",")]
    cuda = not args.emul
    if cuda:
        if not torch.cuda.is_available():
            sys.exit("stream_probe: no CUDA device (use --emul for a dry run on the emulator library)")
        smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
        kw = dict(device="cuda:0")
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
            uniq = list(ex.map(lambda i: K.cached(f"cfg5_i{i}_l19.naf", lambda: K.cfg5_member(i))[0], range(args.unique)))
        source = f"cfg5_member 0..{args.unique - 1} (level 19, 2-6 Mbp), ready in {time.perf_counter() - t0:.0f} s"
    else:
        from _harness import emul_library
        smi = "none (emulator library on the CPU: no rate is a measurement)"
        kw = dict(device="cpu", _library=emul_library())
        uniq = [K.genome(9000 + i, 20_000 + 5_000 * i, level=3, records=1 + i % 3) for i in range(args.unique)]
        source = "tests/_cases.genome, 20-35 kbp, level 3"
    order = [i % len(uniq) for i in range(args.archives)]
    datas = [uniq[u] for u in order]
    sizes = [len(d) for d in datas]
    cuts = cuts_of(sizes, args.batch_bytes)

    # warm-up + parity: every arm's sub-batch exports against the serial arm's
    drop_pool()
    _, ref = run_serial(datas, cuts, kw, cuda, check=True)
    for lanes in lanes_list:
        _, got = run_stream(datas, args.batch_bytes, lanes, kw, cuda, check=True)
        assert got == ref, f"lanes={lanes}: the stream's exports differ from the serial arm's"
    _, lens = run_serial(datas, cuts, kw, cuda)
    ascii_bytes = sum(lens)
    pinned = [torch.frombuffer(bytearray(u), dtype=torch.uint8).pin_memory() for u in uniq] if cuda else None
    if cuda:
        run_h2d(pinned, order, cuts, sizes)

    times = {"serial": [], **{f"lanes_{L}": [] for L in lanes_list}, "h2d": []}
    mem = {k: {"peak_torch_allocated_bytes": 0, "peak_outside_torch_bytes": 0} for k in times}

    def note(name, arm):
        times[name].append(arm.seconds)
        if cuda:
            m = mem[name]
            m["peak_torch_allocated_bytes"] = max(m["peak_torch_allocated_bytes"], arm.peak_torch)
            m["peak_outside_torch_bytes"] = max(m["peak_outside_torch_bytes"], arm.peak_outside)

    for r in range(args.rounds):
        drop_pool()
        note("serial", run_serial(datas, cuts, kw, cuda)[0])
        drop_pool()
        for lanes in (lanes_list if r % 2 == 0 else lanes_list[::-1]):
            note(f"lanes_{lanes}", run_stream(datas, args.batch_bytes, lanes, kw, cuda)[0])
        if cuda:
            note("h2d", run_h2d(pinned, order, cuts, sizes))

    h2d_s = statistics.median(times["h2d"]) if times["h2d"] else None
    arms = {}
    for name, ts in times.items():
        if not ts:
            continue
        s = statistics.median(ts)
        arms[name] = {"seconds": ts, "median_s": s, "ascii_GBps": ascii_bytes / s / 1e9,
                      "frac_of_h2d_ceiling": (h2d_s / s) if h2d_s else None, **(mem[name] if cuda else {})}
    arms["h2d"] = arms.get("h2d", {"not_measured": "no CUDA device"})
    if cuda:
        arms["h2d"]["compressed_GBps"] = sum(sizes) / h2d_s / 1e9
    result = {"probe": "stream_probe", "gpu": smi, "library": "emulator" if args.emul else "libnafgpu.so (sm_100a)",
              "collection": source, "archives": args.archives, "unique": len(uniq), "compressed_bytes": sum(sizes),
              "ascii_bytes": ascii_bytes, "batch_bytes": args.batch_bytes, "sub_batches": len(cuts), "rounds": args.rounds,
              "arms": arms}
    for name, a in arms.items():
        if "median_s" in a:
            print(f"{name:>8}: {a['median_s'] * 1e3:9.1f} ms  {a['ascii_GBps']:8.2f} GB/s ASCII"
                  + (f"  {100 * a['frac_of_h2d_ceiling']:5.1f} % of h2d" if a["frac_of_h2d_ceiling"] else ""), file=sys.stderr)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
