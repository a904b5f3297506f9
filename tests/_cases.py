"""Parity archives produced by the oracle's restatement of the reference encoder (deterministic)."""
import os
import struct
import tempfile
import time

import numpy as np

import _oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TREE_CACHE = os.path.join(ROOT, "bench_cache")
# Per user: on a shared host another user's cache directory would be unwritable, and its archives not ours to trust.
CACHE = os.environ.get("NAFBENCH_CACHE") or os.path.join(tempfile.gettempdir(), f"nafbench_cache_{os.getuid()}")


def cached(name, make):
    """(archive, where it came from).  Archives that take minutes to generate (250 Mbp at zstd level 19: ~3 min on one core)
    are read from bench_cache/ in the tree when someone put them there, else from CACHE, else generated into CACHE.  A new
    file is written under a temporary name and renamed, so an interrupted run leaves no truncated archive behind."""
    for d in (TREE_CACHE, CACHE):
        path = os.path.join(d, name)
        if os.path.exists(path):
            with open(path, "rb") as f:
                return f.read(), f"cached ({os.path.relpath(path, ROOT) if d == TREE_CACHE else path})"
    t0 = time.perf_counter()
    data = make()
    os.makedirs(CACHE, exist_ok=True)
    tmp = os.path.join(CACHE, f"{name}.{os.getpid()}.tmp")
    with open(tmp, "wb") as f:
        f.write(data)
    os.replace(tmp, os.path.join(CACHE, name))
    return data, f"generated in {time.perf_counter() - t0:.0f} s"


def _rng(seed):
    return np.random.default_rng(seed)


def random_dna(rng, n, alphabet=b"ACGT"):
    return bytes(rng.choice(np.frombuffer(alphabet, np.uint8), size=n).astype(np.uint8))


def reference_roundtrip_records():
    # nafcodec/tests/encoder.rs:12-29
    return dict(ids=[b"r1", b"r2"], comments=[b"record 1", b"record 2"],
                sequences=[b"NGCTCTTAAACCTGCTA", b"NTAATAAGCAATGACGGCAGC"],
                qualities=[b"#8CCCGGGGGGGGGGGG", b"#8AACCFF<FFGGFGE@@@@@"])


def multi_record_dna(seed, n_records, max_len, level=3, flush=True, mask=True, empty_every=0):
    rng = _rng(seed)
    lens = rng.integers(0, max_len + 1, size=n_records)
    if empty_every:
        lens[::empty_every] = 0
    seqs = [random_dna(rng, int(l), b"ACGTACGTACGTACGTNRYKM-") for l in lens]
    ids = [b"seq%d" % i for i in range(n_records)]
    coms = [b"comment number %d of the archive" % i if i % 3 else b"" for i in range(n_records)]
    total = int(lens.sum())
    runs = None
    if mask and total:
        runs = []
        s = 0
        while s < total:
            r = int(rng.choice([0, 1, 2, 3, 17, 254, 255, 256, 510, 1000])) if rng.random() < 0.5 else int(rng.integers(0, 400))
            r = min(r, total - s)
            runs.append(r)
            s += r
        if rng.random() < 0.5:
            runs.append(12345)          # trailing run past the end is legal
    return O.encode(ids=ids, comments=coms, sequences=seqs, mask_runs_=runs, level=level, flush_per_record=flush)


def fastq_reads(seed, n_reads, read_len=150, level=0, with_mask=False):
    # cfg4 shape: reads sampled from a small genome, 1% substitutions, N at 1e-3; quality from a 4-symbol Markov chain
    rng = _rng(seed)
    genome = random_dna(rng, 5386)
    g = np.frombuffer(genome, np.uint8)
    seqs, quals, ids = [], [], []
    qsym = np.frombuffer(b"F:,#", np.uint8)
    for i in range(n_reads):
        p = int(rng.integers(0, len(g) - read_len))
        r = g[p:p + read_len].copy()
        sub = rng.random(read_len) < 0.01
        r[sub] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=int(sub.sum()))
        r[rng.random(read_len) < 1e-3] = ord("N")
        seqs.append(r.tobytes())
        st = np.zeros(read_len, np.int64)
        jump = rng.random(read_len) < 0.1
        st[jump] = rng.integers(0, 4, size=int(jump.sum()))
        st = np.maximum.accumulate(np.where(jump, np.arange(read_len), 0))
        q = qsym[(rng.integers(0, 4, size=read_len))[st] % 4]
        quals.append(q.tobytes())
        ids.append(b"SRR0000001.%d" % (i + 1))
    runs = None
    if with_mask:
        total = n_reads * read_len
        runs = O.synth_mask(seed, total, 700.0, 40.0, False)
    return O.encode(ids=ids, sequences=seqs, qualities=quals, mask_runs_=runs, level=level, flush_per_record=True)


def genome(seed, n, level=19, gaps=0, gap_len=0, telomere=0, mask=True, records=1, mean_u=2000.0, mean_m=300.0):
    seq = O.synth_dna(seed, n, gc=0.5, families=2, repeat_len=min(5000, max(n // 50, 10)), copies=7, iupac_rate=1e-5,
                      gap_count=gaps, gap_len=gap_len, telomere=telomere)
    runs = O.synth_mask(seed, n, mean_u, mean_m, True) if mask else None
    if records == 1:
        seqs = [seq]
    else:
        cuts = sorted(set(int(x) for x in _rng(seed).integers(1, n, size=records - 1)))
        cuts = [0] + cuts + [n]
        seqs = [seq[cuts[i]:cuts[i + 1]] for i in range(len(cuts) - 1)]
    ids = [b"synth_%d_%d" % (seed, i) for i in range(len(seqs))]
    coms = [b"synthetic"] * len(seqs)
    return O.encode(ids=ids, comments=coms, sequences=seqs, mask_runs_=runs, level=level, flush_per_record=True)


def text_archive(seqs, sequence_type=O.TEXT, mask_runs=None, level=3, qualities=None):
    ids = [b"t%d" % i for i in range(len(seqs))]
    return O.encode(ids=ids, sequences=seqs, qualities=qualities, mask_runs_=mask_runs, sequence_type=sequence_type, level=level)


def crafted_lengths_archive(words: bytes, ids):
    """Archive with flags Id|Length whose Length section holds `words` verbatim (continuation words, reader.rs:46-68)."""
    body = O.encode(ids=ids)
    L = O.parse(body)
    ids_sec = body[L.sec[0].offset:L.sec[0].offset + L.sec[0].compressed_size]
    q = O.encode(sequence_type=O.TEXT, sequences=[words])
    Lq = O.parse(q)
    frame = q[Lq.sec[4].offset:Lq.sec[4].offset + Lq.sec[4].compressed_size]
    hdr = bytes([0x01, 0xF9, 0xEC, 0x01, 0x28, 0x20]) + O.write_variable_length(60) + O.write_variable_length(len(ids))
    return (hdr + O.write_variable_length(L.sec[0].original_size) + O.write_variable_length(len(ids_sec)) + ids_sec
            + O.write_variable_length(len(words)) + O.write_variable_length(len(frame)) + frame)


def zstd_frame(payload: bytes, level=3, flush_every=0):
    """A magicless zstd frame of `payload`, cut out of a TEXT archive made by the oracle encoder."""
    if flush_every:
        chunks = [payload[i:i + flush_every] for i in range(0, len(payload), flush_every)] or [b""]
    else:
        chunks = [payload]
    arc = O.encode(sequence_type=O.TEXT, sequences=chunks, level=level, flush_per_record=True)
    L = O.parse(arc)
    s = L.sec[4]
    return arc[s.offset:s.offset + s.compressed_size]


# ---- BASELINE.json configs at their stated sizes (SURVEY 8d); shared by bench.py and the slow -m gpu parity tests ------
def cfg3_chromosome(n=250_000_000, seed=3, level=19, workers=None):
    """One record of n residues: N telomeres / centromere / gaps, a diverged 300 bp repeat family, ~50 % soft-masked with mean
    run 300; every section one zstd frame at `level`.  `workers` > 0 lets libzstd compress that one frame on several threads
    (generator convenience: the 125 MB packed stream takes minutes on one core); the reference's call pattern is workers=0."""
    import os
    seq = O.synth_chromosome(seed, n)
    runs = O.synth_mask(seed, n, 300.0, 300.0, True)
    off = np.array([0, n], dtype=np.uint64)
    O.set_encoder_workers(min(os.cpu_count() or 1, 16) if workers is None else workers)
    try:
        return O.encode_blobs(1, ids=(np.frombuffer(b"synth_chr", np.uint8), np.array([0, 9], np.uint64)),
                              comments=(np.frombuffer(b"synthetic", np.uint8), np.array([0, 9], np.uint64)),
                              sequences=(seq, off), mask_runs_=runs, level=level, flush_per_record=True)
    finally:
        O.set_encoder_workers(0)


def cfg4_fastq(n_reads=1_000_000, seed=4, read_len=150, level=0, with_mask=True):
    """n_reads x read_len FASTQ in the reference encoder's framing (a zstd flush after every record: one tiny block per read
    and stream, encoder/mod.rs:271,298,319), flags Id|Length|Sequence|Quality (+ Mask), level = the reference default."""
    ids, ids_off, seq, qual = O.synth_fastq(seed, n_reads, read_len)
    off = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(read_len)
    runs = O.synth_mask(seed, n_reads * read_len, 700.0, 40.0, False) if with_mask else None
    return O.encode_blobs(n_reads, ids=(ids, ids_off), sequences=(seq, off), qualities=(qual, off), mask_runs_=runs, level=level,
                          flush_per_record=True)


def cfg5_member(i, base_seed=5000, level=19):
    """Archive i of the RefSeq-collection shape: the cfg2 generator with seed base + i, N uniform in [2, 6] Mbp, one
    chromosome + 0-3 plasmid records."""
    rng = _rng(base_seed + i)
    n = int(rng.integers(2_000_000, 6_000_001))
    plasmids = int(rng.integers(0, 4))
    seq = O.synth_dna(base_seed + i, n, gc=0.5, families=2, repeat_len=5000, copies=7, iupac_rate=1e-5)
    runs = O.synth_mask(base_seed + i, n, 2000.0, 300.0, True)
    cuts = [0] + sorted(n - int(x) for x in rng.integers(3_000, 200_000, size=plasmids).cumsum()) + [n] if plasmids else [0, n]
    seqs = [seq[cuts[k]:cuts[k + 1]] for k in range(len(cuts) - 1)]
    ids = [b"synth_%d_%d" % (base_seed + i, k) for k in range(len(seqs))]
    return O.encode(ids=ids, comments=[b"synthetic"] * len(seqs), sequences=seqs, mask_runs_=runs, level=level, flush_per_record=True)
