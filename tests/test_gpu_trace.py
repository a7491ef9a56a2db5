"""-m gpu: trace points -> edit scripts (fgb_compute_trace_pts, SURVEY row a-17) against the
UNMODIFIED reference's Compute_Trace_PTS on the alignments the path itself emits: same int script,
same diffs, for every record (the reference's scripts are stored by tests/golden/make_golden.py)."""
import hashlib

import numpy as np
import pytest

import oracle_lib as ol
from fastga_b200 import formats, lib, synth

pytestmark = pytest.mark.gpu


def trace_pair(seed, total, ncontig, div, sv, flip=()):
    A, B = synth.make_pair(seed, total, ncontig, div, sv_every=sv)
    for i in flip:                                   # whole contigs on the opposite strand
        B[i] = (3 - B[i][::-1]).astype(np.uint8)
    return formats.genome_from_arrays(A), formats.genome_from_arrays(B)


TRACE_PAIRS = {"5pct": (21, 3_000_000, 4, 0.05, 60_000), "15pct_both_strands": (22, 2_000_000, 5, 0.15, 30_000, (0, 3))}


def _check_pair(name):
    """the reference's Compute_Trace_PTS(aln, work, 100, GREEDIEST, 1, -1), as ALNtoPAF.c:251-272
    calls it, on the same alignments: per record its diffs, script length and script md5
    (tests/golden/reference_runs.json)"""
    gA, gB = trace_pair(*TRACE_PAIRS[name])
    alns, _ = lib.fastga(gA, gB)
    assert len(alns) > 0
    dA, dB = lib.DeviceGenome(gA), lib.DeviceGenome(gB, want_revcomp=True)
    soff, script, diffs = lib.compute_trace_pts(dA, dB, alns)
    want = {tuple(r[:7]): r[7:] for r in ol.reference_run("trace/" + name)["scripts"]}
    assert len(want) == len(alns)
    assert (diffs >= 0).all()
    ncomp = 0
    for i in range(len(alns)):
        key = tuple(int(x) for x in alns.fields[i, :7])
        df, slen, md5 = want[key]
        got = np.ascontiguousarray(script[soff[i]:soff[i + 1]], dtype=np.int32)
        assert df == diffs[i], (i, df, int(diffs[i]))
        assert len(got) == slen and hashlib.md5(got.tobytes()).hexdigest() == md5, (i, got[:8])
        ncomp += int(alns.fields[i, 0])
    return len(alns), ncomp


def test_scripts_match_reference_5pct():
    n, ncomp = _check_pair("5pct")
    assert n > 10


def test_scripts_match_reference_15pct_both_strands():
    n, ncomp = _check_pair("15pct_both_strands")
    assert n > 10 and ncomp > 0


def test_inconsistent_trace_points_are_flagged_not_fatal():
    A, B = synth.make_pair(23, 600_000, 2, 0.05, sv_every=50_000)
    gA, gB = formats.genome_from_arrays(A), formats.genome_from_arrays(B)
    alns, _ = lib.fastga(gA, gB)
    dA, dB = lib.DeviceGenome(gA), lib.DeviceGenome(gB, want_revcomp=True)
    i = int(np.argmax(alns.fields[:, 8]))
    alns.pool[int(alns.toff[i]) + 2] = 0          # claim zero differences in a tile that has some
    alns.pool[int(alns.toff[i]) + 4] = 0
    alns.pool[int(alns.toff[i]) + 6] = 0
    soff, script, diffs = lib.compute_trace_pts(dA, dB, alns)
    good = [k for k in range(len(alns)) if k != i]
    assert (diffs[good] >= 0).all()
    assert diffs[i] == -1 or diffs[i] >= 0        # only flagged when a tile really cannot be aligned
