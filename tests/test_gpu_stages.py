"""-m gpu: every CUDA stage against the oracle on the same seeded input, through the C-ABI."""
import numpy as np
import pytest

import oracle_lib as ol
from fastga_b200 import formats, lib, synth

pytestmark = pytest.mark.gpu


def test_sort128_matches_stable_numpy_sort():
    rng = np.random.default_rng(5)
    for n in (0, 1, 31, 4096, 4097, 100_003, 1_500_000):
        recs = rng.integers(0, 1 << 63, size=(n, 2), dtype=np.uint64)
        recs[:, 1] &= np.uint64(0xffff)            # many equal high keys -> exercises stability
        recs[:, 0] &= np.uint64(0xffff0000ffffffff)
        want = recs.copy()
        key_hi = want[:, 1]
        key_lo = want[:, 0] >> np.uint64(48)
        order = np.lexsort((key_lo, key_hi))        # lexsort is stable
        want = want[order]
        got = lib.sort128_host(recs.copy(), 6, 16)
        assert np.array_equal(got, want), n


def test_sort128_full_key_random():
    rng = np.random.default_rng(6)
    recs = rng.integers(0, 1 << 63, size=(300_000, 2), dtype=np.uint64)
    got = lib.sort128_host(recs.copy(), 0, 16)
    order = np.lexsort((recs[:, 0], recs[:, 1]))
    assert np.array_equal(got, recs[order])


def test_staged_genome_and_revcomp(small_pair):
    gA, _ = small_pair
    dg = lib.DeviceGenome(gA, want_revcomp=True)
    words, woff = dg.download(False)
    rwords, _ = dg.download(True)
    for c in range(gA.ncontig):
        a = gA.contig(c)
        n = len(a)
        w = words[woff[c]:woff[c + 1]]
        bits = ((w[:, None] >> (np.arange(32, dtype=np.uint64) * np.uint64(2))) & np.uint64(3)).reshape(-1)
        assert np.array_equal(bits[:n].astype(np.uint8), a)
        assert not bits[n:].any()
        rw = rwords[woff[c]:woff[c + 1]]
        rbits = ((rw[:, None] >> (np.arange(32, dtype=np.uint64) * np.uint64(2))) & np.uint64(3)).reshape(-1)
        assert np.array_equal(rbits[:n].astype(np.uint8), (3 - a[::-1]))
        assert not rbits[n:].any()


def test_gix_build_matches_oracle(small_pair):
    for g in small_pair:
        dg = lib.DeviceGenome(g)
        perm, rank = ol.contig_rank(g.clen)
        assert np.array_equal(dg.perm, perm)
        want, wstart = ol.gix_build(g, rank)
        gx = lib.DeviceGix.build(dg)
        tab, pstart, _ = gx.download()
        assert gx.n == len(want)
        assert np.array_equal(tab, want)
        assert np.array_equal(pstart, wstart)


def test_gix_build_with_heavy_repeats_matches_oracle():
    """exact tandem repeats put > 4096 records into one 16-bit prefix bin: the oversized-bin path
    of the bucketed k-mer sort (compaction + generic sort + copy back) and the packed groups"""
    rng = np.random.default_rng(77)
    unit = rng.integers(0, 4, 37, dtype=np.uint8)
    contigs = [rng.integers(0, 4, 300_000, dtype=np.uint8), np.tile(unit, 8000),
               np.zeros(50_000, dtype=np.uint8), rng.integers(0, 4, 150_001, dtype=np.uint8)]
    g = formats.genome_from_arrays(contigs)
    dg = lib.DeviceGenome(g)
    perm, rank = ol.contig_rank(g.clen)
    want, wstart = ol.gix_build(g, rank)
    gx = lib.DeviceGix.build(dg)
    tab, pstart, _ = gx.download()
    assert gx.n == len(want)
    assert np.array_equal(tab, want)
    assert np.array_equal(pstart, wstart)


def _share_from_records(g, full, lo, hi, seed):
    """one rank's slice of a k-mer-space sharded table the way the sharded path builds it
    (fgb_gix_from_records): the rows of the full table whose 12-base prefix lies in [lo, hi), in a
    seeded random order on the device"""
    import torch
    rows = full[((full[:, 1] >> np.uint64(40)) >= lo) & ((full[:, 1] >> np.uint64(40)) < hi)]
    rows = rows[np.random.default_rng(seed).permutation(len(rows))]
    recs = torch.from_numpy(rows.view(np.int64).copy()).cuda()
    pb, cb = formats.gix_bytes(g)
    return lib.gix_from_records(recs.data_ptr() if len(rows) else 0, len(rows), lo, hi, False, pb, cb, g.ncontig)


@pytest.mark.parametrize("target", ["8", "1"])
def test_gix_with_more_than_65536_bins_is_the_same_table_whole_and_from_records(small_pair, target):
    """tables beyond ~100 M records are partitioned into more than 2^16 prefix bins (a third, narrower
    digit pass) so that a bin still fits a CTA's shared memory; FGB_KSORT_BIN_TARGET forces that regime
    on a small table (2^19 .. 2^22 bins here), whole table and shares alike"""
    import os
    g = small_pair[1]
    dg = lib.DeviceGenome(g)
    full, pstart, _ = lib.DeviceGix.build(dg).download()
    os.environ["FGB_KSORT_BIN_TARGET"] = target
    try:
        tab2, pstart2, _ = lib.DeviceGix.build(dg).download()
        parts = [_share_from_records(g, full, lo, hi, k).download()[0]
                 for k, (lo, hi) in enumerate(((0, (1 << 23) + 5), ((1 << 23) + 5, 1 << 24)))]
    finally:
        del os.environ["FGB_KSORT_BIN_TARGET"]
    assert np.array_equal(tab2, full) and np.array_equal(pstart2, pstart)
    assert np.array_equal(np.concatenate(parts), full)


def test_gix_slices_from_records_concatenate_to_the_full_table(small_pair):
    """one rank's slice of a k-mer-space sharded table (fgb_gix_from_records) is binned relative to
    its own prefix range; uneven shares must concatenate to exactly the single-GPU table"""
    g = small_pair[1]
    dg = lib.DeviceGenome(g)
    full, _, _ = lib.DeviceGix.build(dg).download()
    cuts = [0, 1 << 21, (1 << 23) + 12345, (3 << 22) + 7, 1 << 24]
    parts = []
    for k, (lo, hi) in enumerate(zip(cuts[:-1], cuts[1:])):
        sh = _share_from_records(g, full, lo, hi, k)
        tab = sh.download()[0]
        assert len(tab) == sh.n
        if sh.n:
            pre = (tab[:, 1] >> np.uint64(40)).astype(np.int64)
            assert pre.min() >= lo and pre.max() < hi
        parts.append(tab)
    assert np.array_equal(np.concatenate(parts), full)


def test_merge_and_seed_sort_match_oracle(small_pair):
    gA, gB = small_pair
    dA, dB = lib.DeviceGenome(gA), lib.DeviceGenome(gB)
    xA, xB = lib.DeviceGix.build(dA), lib.DeviceGix.build(dB)
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    ds = lib.DeviceSeeds.find(xA, xB, amx, bmx, 10)
    tA, _, _ = xA.download(False)
    tB, pB, _ = xB.download()
    seeds, sumlen = ol.merge(tA, tB, pB, 10)
    assert ds.n == len(seeds) and ds.sumlen == sumlen
    want = ol.seed_records(seeds, ds.layout + (amx, bmx), sort=True)
    got = ds.download()
    assert np.array_equal(got, want)


@pytest.mark.parametrize("copies", [2, 5])
def test_merge_against_a_denser_second_table(copies):
    """a shard of genome 1 against all of genome 2 (multi-GPU): T2 is several times denser than T1,
    the merge switches to 32- / 16-entry tiles so that the block's T2 slice still fits its staging"""
    rng = np.random.default_rng(90 + copies)
    a = rng.integers(0, 4, 400_000, dtype=np.uint8)
    B = [synth.diverged_copy(rng, a, 0.03 + 0.01 * k, sv_every=60_000) for k in range(copies)]
    B = [b[:len(b) - 7 * k] for k, b in enumerate(B)]
    gA, gB = formats.genome_from_arrays([a]), formats.genome_from_arrays(B)
    dA, dB = lib.DeviceGenome(gA), lib.DeviceGenome(gB)
    xA, xB = lib.DeviceGix.build(dA), lib.DeviceGix.build(dB)
    assert xB.n > 1.6 * xA.n
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    ds = lib.DeviceSeeds.find(xA, xB, amx, bmx, 10)
    tA, _, _ = xA.download(False)
    tB, pB, _ = xB.download()
    seeds, sumlen = ol.merge(tA, tB, pB, 10)
    assert ds.n == len(seeds) and ds.sumlen == sumlen
    want = ol.seed_records(seeds, ds.layout + (amx, bmx), sort=True)
    assert np.array_equal(ds.download(), want)


def test_forward_only_table_is_the_forward_subset_and_merges_identically(small_pair):
    """the fused path builds the adaptamer side forward-strand-only (fgb_gix_build_forward): the table
    must be exactly the forward entries of the both-strand table, in order, and seed identically"""
    gA, gB = small_pair
    dA, dB = lib.DeviceGenome(gA), lib.DeviceGenome(gB)
    xA, xF, xB = lib.DeviceGix.build(dA), lib.DeviceGix.build_forward(dA), lib.DeviceGix.build(dB)
    tA, pA, _ = xA.download()
    tF, pF, _ = xF.download()
    fwd = ((tA[:, 0] >> np.uint64(47)) & np.uint64(1)) == 0
    assert np.array_equal(tF, tA[fwd])
    pre = (tF[:, 1] >> np.uint64(40)).astype(np.int64)
    assert np.array_equal(pF.astype(np.int64), np.searchsorted(pre, np.arange((1 << 24) + 1)))
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    s1 = lib.DeviceSeeds.find(xA, xB, amx, bmx, 10)
    s2 = lib.DeviceSeeds.find(xF, xB, amx, bmx, 10)
    assert s1.n == s2.n and s1.sumlen == s2.sumlen
    assert np.array_equal(s1.download(), s2.download())


def test_merge_with_repeats_takes_the_unstaged_and_the_crowded_paths():
    """long exact repeats: (1) a T1 tile whose T2 slice exceeds the staging buffer (searched straight
    from HBM), (2) a tile with more seeds than descriptors at a high -f (entry-wise write-out);
    both must equal the oracle's state machine"""
    rng = np.random.default_rng(123)
    unit = rng.integers(0, 4, 997, dtype=np.uint8)
    a = np.concatenate([rng.integers(0, 4, 100_000, dtype=np.uint8), np.tile(unit, 100),
                        np.zeros(60, dtype=np.uint8), rng.integers(0, 4, 50_000, dtype=np.uint8)])
    b = np.concatenate([rng.integers(0, 4, 50_000, dtype=np.uint8), np.tile(unit, 40),
                        np.zeros(3000, dtype=np.uint8),
                        synth.diverged_copy(rng, a[:100_000], 0.04, sv_every=50_000)])
    gA, gB = formats.genome_from_arrays([a]), formats.genome_from_arrays([b])
    dA, dB = lib.DeviceGenome(gA), lib.DeviceGenome(gB)
    xA, xB = lib.DeviceGix.build(dA), lib.DeviceGix.build(dB)
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    tA, _, _ = xA.download(False)
    tB, pB, _ = xB.download()
    for freq in (3, 10, 64, 200, 255):
        ds = lib.DeviceSeeds.find(xA, xB, amx, bmx, freq)
        seeds, sumlen = ol.merge(tA, tB, pB, freq)
        assert ds.n == len(seeds) and ds.sumlen == sumlen, freq
        want = ol.seed_records(seeds, ds.layout + (amx, bmx), sort=True)
        assert np.array_equal(ds.download(), want), freq


def _canon(recs, pool, aread=None, bread=None, comp=None):
    out = []
    for i, r in enumerate(recs):
        tr = bytes(pool[int(r["toff"]):int(r["toff"]) + int(r["tlen"])])
        out.append((int(comp[i]) if comp is not None else int(r["comp"]),
                    int(aread[i]) if aread is not None else int(r["aread"]),
                    int(bread[i]) if bread is not None else int(r["bread"]),
                    int(r["abpos"]), int(r["bbpos"]), int(r["aepos"]), int(r["bepos"]), int(r["diffs"]), tr))
    return out


def test_extend_matches_oracle(small_pair):
    gA, gB = small_pair
    dA, dB = lib.DeviceGenome(gA, want_revcomp=True), lib.DeviceGenome(gB)
    xA, xB = lib.DeviceGix.build(dA), lib.DeviceGix.build(dB)
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    ds = lib.DeviceSeeds.find(xA, xB, amx, bmx, 10)
    seeds = ds.download()
    layout = ds.layout + (amx, bmx)
    want, wpool, whits = ol.search(seeds, layout, gA, gB, dA.perm, dB.perm, gA.freq)
    ov = lib.DeviceOverlaps.extend(ds, dA, dB, gA.freq)
    got, gpool = ov.records()
    cnt = ov.counters()
    assert cnt["hits"] == whits
    # pairkey = (comp, icont rank, jcont rank) packed as in the seed record
    jb, ib = layout[2], layout[3]
    pk = got["pairkey"].astype(np.int64)
    jc = pk & ((1 << jb) - 1)
    ic = (pk >> jb) & ((1 << ib) - 1)
    comp = pk >> (jb + ib)
    g = _canon(got, gpool, dA.perm[ic], dB.perm[jc], comp)
    w = _canon(want, wpool)
    assert len(g) == len(w)
    assert g == w          # same records in the same (reference discovery) order


# ---------------------------------------------------------------------------------------------
#  the reference's extern sort seams (msd_sort / rmsd_sort) against what libfastga_ref.so returned
#  on the same inputs (tests/golden/reference_runs.json)
# ---------------------------------------------------------------------------------------------

import ctypes as C
import hashlib


class _Range(C.Structure):
    _fields_ = [("beg", C.c_int), ("end", C.c_int), ("off", C.c_int64)]


MSD_ARGTYPES = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
RMSD_ARGTYPES = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]


def msd_input():
    """records in GIXmake's shape on EXAMPLE (swide 15, KBYTES 10): (array + 16 pad bytes, n, rsize,
    ksize, part, beg, end)"""
    rng = np.random.default_rng(9)
    rsize, ksize, beg, end = 15, 10, 3, 40
    counts = rng.integers(0, 3000, end - beg)
    counts[5] = 0
    n = int(counts.sum())
    arr = rng.integers(0, 256, (n, rsize), dtype=np.uint8)
    arr[:, 0] = 0
    arr[:, 3:9] &= 0x03                              # few distinct keys -> long equal runs and LCPs
    part = np.zeros(1024, dtype=np.int64)
    part[beg:end] = counts * rsize
    return np.concatenate([arr.reshape(-1), np.zeros(16, np.uint8)]), n, rsize, ksize, part, beg, end


def msd_payload_md5(r, ksize):
    """payloads of the sorted records with every equal-key run put in order (the sort is not stable)"""
    n, rsize = r.shape
    run = np.cumsum(r[:, 0] != 0)
    pay = np.zeros(n, dtype=np.uint64)
    for k in range(ksize, rsize):
        pay |= r[:, k].astype(np.uint64) << np.uint64(8 * (k - ksize))
    return hashlib.md5(pay[np.lexsort((pay, run))].tobytes()).hexdigest()


def test_msd_sort_seam_matches_reference():
    from fastga_b200 import load_library
    L = load_library()
    a, n, rsize, ksize, part, beg, end = msd_input()
    L.fgb_msd_sort.argtypes = MSD_ARGTYPES
    L.fgb_msd_sort(a.ctypes.data, n, rsize, ksize, part.ctypes.data, beg, end, 4)
    want = ol.reference_run("seam/msd_sort")
    r = a[:n * rsize].reshape(n, rsize)
    assert a[n * rsize] == want["sentinel"] == 1
    # LCP byte + key bytes identical, payloads the same multiset per equal-key run
    assert hashlib.md5(np.ascontiguousarray(r[:, :ksize]).tobytes()).hexdigest() == want["keys_md5"]
    assert msd_payload_md5(r, ksize) == want["payload_md5"]


def rmsd_input():
    """FastGA's seed record on EXAMPLE (swide 9): (array, n, rsize, nparts, part, nthreads)"""
    rng = np.random.default_rng(10)
    rsize, nparts, nthreads = 9, 37, 8
    counts = rng.integers(0, 5000, nparts)
    counts[[0, 7]] = 0
    n = int(counts.sum())
    arr = rng.integers(0, 256, (n, rsize), dtype=np.uint8)
    arr[:, 5:] &= 0x07
    part = (counts * rsize).astype(np.int64)
    return arr.reshape(-1).copy(), n, rsize, nparts, part, nthreads


def test_rmsd_sort_seam_matches_reference():
    from fastga_b200 import load_library
    L = load_library()
    a, n, rsize, nparts, part, nthreads = rmsd_input()
    p = (_Range * nthreads)()
    L.fgb_rmsd_sort.argtypes = RMSD_ARGTYPES
    n2 = L.fgb_rmsd_sort(a.ctypes.data, n, rsize, rsize, nparts, part.ctypes.data, nthreads, p)
    want = ol.reference_run("seam/rmsd_sort")
    assert [[p[i].beg, p[i].end, p[i].off] for i in range(n2)] == want["ranges"]
    assert hashlib.md5(a.tobytes()).hexdigest() == want["md5"]
