"""BASELINE.json configs at their STATED sizes, bit-exact against the oracle on the device (`-m gpu`, slow-marked).

These reach code paths only large inputs do: the 15 000-chunk carry loop of k_unpack and the sliced mask scan (250 Mbp),
multi-wave LZ finisher and `fin_g` at 4 B per byte, the 2 x 10^6-block frame scan and worklists (10^6 reads), and a
collection job of many unequal archives.  The 250 Mbp archive takes ~3 min to generate at zstd level 19 on one core; it
is kept in the archive cache that bench.py shares (tests/_cases.py: cached)."""
import hashlib
import os

import numpy as np
import pytest

import _cases as K
import _oracle as O
import nafcodec_b200 as N
from _harness import assert_same_as_oracle, cuda_library

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


def test_cfg3_250mbp_single_frame():
    lib = cuda_library()
    data = K.cached("cfg3_n250000000_s3_l19.naf", lambda: K.cfg3_chromosome(250_000_000, workers=0))[0]
    L = O.parse(data)
    assert L.sec[4].original_size == 250_000_000 and L.number_of_sequences == 1
    res = N.shared_context(0, lib).decode([N.parse_archive(data, lib)])[0]
    want = O.decode(data)
    assert_same_as_oracle(res, want, "cfg3 250 Mbp")
    # size-independent properties: residue census of the generator's shape and the lower-case share of a ~50 % mask
    a = np.frombuffer(res.sequence, np.uint8)
    assert len(a) == 250_000_000
    assert hashlib.sha256(res.sequence).digest() == hashlib.sha256(want.sequence).digest()
    lower = int((a >= 97).sum())
    n_count = int(((a | 0x20) == ord("n")).sum())
    assert 0.40 < lower / len(a) < 0.60
    assert n_count >= 3_000_000 + 20 * 50_000 - 100_000          # centromere + gaps (gaps may overlap) + telomeres
    # the same archive without the mask is the upper-cased sequence
    up = N.shared_context(0, lib).decode([N.parse_archive(data, lib)], N.decoder._want_bits(True, True, True, True, False))[0]
    assert np.array_equal(np.frombuffer(up.sequence, np.uint8), np.where((a >= 97) & (a <= 122), a - 32, a))


@pytest.mark.parametrize("quality", [True, False])
def test_cfg4_million_reads(quality):
    lib = cuda_library()
    data = K.cfg4_fastq(1_000_000)
    L = O.parse(data)
    assert L.number_of_sequences == 1_000_000 and L.flags & 0x01
    want_bits = N.decoder._want_bits(True, True, True, quality, True)
    res = N.shared_context(0, lib).decode([N.parse_archive(data, lib)], want_bits)[0]
    want = O.decode(data, quality=quality)
    assert_same_as_oracle(res, want, f"cfg4 1M reads quality={quality}")
    assert res.n_lengths == 1_000_000 and int(res.lengths.min()) == 150 and int(res.lengths.max()) == 150
    assert (res.quality is None) == (not quality)
    st = N.shared_context(0, lib).stats()
    assert st.n_blocks > (2_000_000 if quality else 1_000_000)    # one tiny zstd block per read and flushed stream


def test_cfg5_collection_mix():
    lib = cuda_library()
    from concurrent.futures import ThreadPoolExecutor
    n = 64
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        arcs = list(ex.map(lambda i: K.cached(f"cfg5_i{i}_l19.naf", lambda: K.cfg5_member(i))[0], range(n)))
        wants = list(ex.map(O.decode, arcs))
    res = N.decode_batch(arcs, _library=lib)
    sizes = set()
    for i, (r, w) in enumerate(zip(res, wants)):
        assert_same_as_oracle(r, w, f"cfg5 archive {i}")
        sizes.add(r.total_residues)
        assert 2_000_000 <= r.total_residues <= 6_000_000 and 1 <= r.n_records <= 4
    assert len(sizes) == n
