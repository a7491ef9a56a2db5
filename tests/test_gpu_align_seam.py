"""-m gpu: the align.h seam -- fgb_local_alignments (batched Local_Alignment) against the UNMODIFIED
reference's Local_Alignment on random call tuples, borders included (its results are stored in
tests/golden/reference_paths.npz by tests/golden/make_golden.py)."""
import numpy as np
import pytest

import oracle_lib as ol
from fastga_b200 import formats, lib, synth

pytestmark = pytest.mark.gpu


def seam_jobs(borders):
    """six contigs, their diverged copies and 300 random Local_Alignment call tuples on them:
    (A, B, jobs (i, j, comp, low, hgh, anti, lbord, hbord))"""
    rng = np.random.default_rng(41 + int(borders))
    ncont = 6
    A = [rng.integers(0, 4, int(rng.integers(3000, 40000)), dtype=np.uint8) for _ in range(ncont)]
    B, pad = [], []
    for a in A:
        rate = float(rng.choice([0.02, 0.05, 0.1, 0.15]))
        b = synth.diverged_copy(rng, a, rate, sv_every=0, inversions=False)      # small mutations only
        pad.append(int(rng.integers(0, 300)))
        B.append(np.concatenate([rng.integers(0, 4, pad[-1], dtype=np.uint8), b]))
    jobs = []
    for _ in range(300):
        i = int(rng.integers(0, ncont))
        comp = int(rng.random() < 0.4)
        la, lb = len(A[i]), len(B[i])
        x = int(rng.integers(100, la - 100))
        y = int(np.clip(x + (lb - la) + int(rng.integers(-60, 60)), 50, lb - 50))
        if comp:                       # the strand-C call sees reverse-complemented A: any diagonal will do
            y = int(rng.integers(50, lb - 50))
        d, anti = x - y, x + y
        low, hgh = d - int(rng.integers(0, 70)), d + int(rng.integers(0, 70))
        lbd = hbd = -1
        if borders:
            lbd = int(rng.integers(0, 40)) if rng.random() < 0.7 else -1
            hbd = int(rng.integers(0, 40)) if rng.random() < 0.7 else -1
        jobs.append((i, i, comp, low, hgh, anti, lbd, hbd))
    return A, B, np.array(jobs, dtype=np.int32)


@pytest.mark.parametrize("borders", [False, True])
def test_batched_local_alignment_matches_reference(borders):
    A, B, jobs = seam_jobs(borders)
    gA, gB = formats.genome_from_arrays(A), formats.genome_from_arrays(B)
    dA, dB = lib.DeviceGenome(gA, want_revcomp=True), lib.DeviceGenome(gB)
    paths, toff, traces = lib.local_alignments(dA, dB, jobs, gA.freq)

    want, wtrace = ol.reference_paths("seam_%s" % borders)
    assert len(want) == len(jobs)
    nonempty = 0
    for q in range(len(jobs)):
        got = paths[q]
        assert got[6] == 0, (q, got)
        assert tuple(int(v) for v in want[q]) == tuple(int(v) for v in got[:6]), (q, jobs[q])
        tlen = int(want[q][5])
        assert np.array_equal(wtrace[q], traces[int(toff[q]):int(toff[q]) + tlen]), q
        nonempty += int(want[q][2] > want[q][0])
    assert nonempty > 100
