"""The host's plan of a job, pinned: which kernels the path choices launch, how many profiled stages there are, how many bytes
cross PCIe each way, and how many frames, blocks and sequences the header walk finds.  Every case runs under each of the test
overrides (NAFGPU_*) that steer those choices, and must still decode what the oracle decodes.

The expected values are literals: the host layer that makes these choices (nafgpu_api.cu, launch_zstd_stage) may be
restructured, but not what it decides.  lz_rounds, lz_flow and lz_handover depend on device-side deadlines and are left out."""
import numpy as np
import pytest

import _cases as K
import _oracle as O
import nafcodec_b200 as N
from _harness import BACKENDS, assert_same_as_oracle, library
from conftest import read_golden
from test_parity import _generations

pytestmark = pytest.mark.parametrize("backend", BACKENDS)

GOLDEN = ["masked.naf", "LuxC.naf", "phix.naf", "CP040672.naf", "NZ_AAEN01000029.naf"]
CASES = GOLDEN + ["batch", "fastq", "frame"]
OVERRIDES = {
    "none": {},
    "lz_small_0": {"NAFGPU_LZ_SMALL": "0"},
    "tiny_0": {"NAFGPU_TINY_BLOCKS": "0"},
    "tiny_1": {"NAFGPU_TINY_BLOCKS": "1"},
    "huf_block_min_1": {"NAFGPU_HUF_BLOCK_MIN": "1"},
    "flow_early_1": {"NAFGPU_LZ_FLOW_EARLY": "1"},
    "fs_tile_37": {"NAFGPU_FS_TILE": "37"},
    "walk_split_3": {"NAFGPU_WALK_SPLIT": "3"},
}
STATS = ("kernel_launches", "n_stages", "h2d_bytes", "d2h_bytes", "n_frames", "n_blocks", "n_sequences")

_inputs = {}


def _input(case):
    """(kind, data) of a case: an archive, a list of archives, or a payload for one zstd frame."""
    if case not in _inputs:
        if case in GOLDEN:
            _inputs[case] = ("archives", [read_golden(case)])
        elif case == "batch":
            _inputs[case] = ("archives", [read_golden("masked.naf"), read_golden("phix.naf")])
        elif case == "fastq":                                      # one tiny block per read and stream
            _inputs[case] = ("archives", [K.fastq_reads(41, 300)])
        else:                                                      # one dependency chain: the finisher takes it over
            p = _generations(np.random.default_rng(7), 3000, 100)
            _inputs[case] = ("frame", (K.zstd_frame(p, 3), p))
    return _inputs[case]


def run_case(backend, case):
    """Decodes the case on the shared context, checks it against the oracle and returns the context."""
    lib = library(backend)
    ctx = N.shared_context(0, lib)
    kind, data = _input(case)
    if kind == "frame":
        frame, p = data
        assert ctx.zstd_decompress(frame, len(p)) == p
    else:
        got = ctx.decode([N.parse_archive(a, lib) for a in data])
        for i, (r, a) in enumerate(zip(got, data)):
            assert_same_as_oracle(r, O.decode(a), f"{case} archive {i}")
    return ctx


# (kernel_launches, n_stages, h2d_bytes, d2h_bytes, n_frames, n_blocks, n_sequences), per (case, override)
EXPECTED = {
    ('masked.naf', 'none'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'lz_small_0'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'tiny_0'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'tiny_1'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'huf_block_min_1'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'flow_early_1'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'fs_tile_37'): (10, 14, 2019, 4560, 5, 5, 0),
    ('masked.naf', 'walk_split_3'): (10, 14, 2019, 4560, 5, 5, 0),
    ('LuxC.naf', 'none'): (13, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'lz_small_0'): (15, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'tiny_0'): (13, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'tiny_1'): (15, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'huf_block_min_1'): (13, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'flow_early_1'): (13, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'fs_tile_37'): (13, 14, 3870, 8264, 4, 4, 278),
    ('LuxC.naf', 'walk_split_3'): (13, 14, 3870, 8264, 4, 4, 278),
    ('phix.naf', 'none'): (14, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'lz_small_0'): (16, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'tiny_0'): (14, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'tiny_1'): (16, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'huf_block_min_1'): (14, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'flow_early_1'): (14, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'fs_tile_37'): (14, 14, 6954, 27864, 6, 6, 571),
    ('phix.naf', 'walk_split_3'): (14, 14, 6954, 27864, 6, 6, 571),
    ('CP040672.naf', 'none'): (14, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'lz_small_0'): (16, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'tiny_0'): (14, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'tiny_1'): (16, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'huf_block_min_1'): (14, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'flow_early_1'): (14, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'fs_tile_37'): (14, 14, 27754, 111184, 5, 5, 719),
    ('CP040672.naf', 'walk_split_3'): (14, 14, 27754, 111184, 5, 5, 719),
    ('NZ_AAEN01000029.naf', 'none'): (12, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'lz_small_0'): (14, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'tiny_0'): (12, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'tiny_1'): (14, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'huf_block_min_1'): (12, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'flow_early_1'): (12, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'fs_tile_37'): (12, 14, 1336012, 5493364, 5, 25, 107),
    ('NZ_AAEN01000029.naf', 'walk_split_3'): (12, 14, 1336012, 5493364, 5, 25, 107),
    ('batch', 'none'): (14, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'lz_small_0'): (16, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'tiny_0'): (14, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'tiny_1'): (16, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'huf_block_min_1'): (14, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'flow_early_1'): (14, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'fs_tile_37'): (14, 14, 8925, 32256, 11, 11, 571),
    ('batch', 'walk_split_3'): (14, 14, 8925, 32256, 11, 11, 571),
    ('fastq', 'none'): (16, 14, 69828, 102216, 4, 604, 4454),
    ('fastq', 'lz_small_0'): (15, 14, 69828, 102216, 4, 604, 4454),
    ('fastq', 'tiny_0'): (16, 14, 69828, 102216, 4, 604, 4454),
    ('fastq', 'tiny_1'): (18, 14, 69828, 102216, 4, 604, 4454),
    ('fastq', 'huf_block_min_1'): (16, 14, 69828, 102216, 4, 604, 4454),
    ('fastq', 'flow_early_1'): (16, 14, 69828, 102216, 4, 604, 4454),
    ('fastq', 'fs_tile_37'): (19, 14, 70148, 102216, 4, 604, 4454),
    ('fastq', 'walk_split_3'): (16, 14, 69828, 102216, 4, 604, 4454),
    ('frame', 'none'): (12, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'lz_small_0'): (11, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'tiny_0'): (12, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'tiny_1'): (14, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'huf_block_min_1'): (12, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'flow_early_1'): (12, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'fs_tile_37'): (12, 14, 9262, 305472, 1, 4, 2921),
    ('frame', 'walk_split_3'): (12, 14, 9262, 305472, 1, 4, 2921),
}


@pytest.mark.parametrize("override", list(OVERRIDES))
@pytest.mark.parametrize("case", CASES)
def test_job_plan(backend, monkeypatch, case, override):
    for k, v in OVERRIDES[override].items():
        monkeypatch.setenv(k, v)
    ctx = run_case(backend, case)
    st = ctx.stats()
    assert tuple(getattr(st, k) for k in STATS) == EXPECTED[(case, override)]
    assert len(ctx.profile_stages()) == st.n_stages
