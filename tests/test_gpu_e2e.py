"""-m gpu: the reference-facing call (fgb_fastga, host buffers) against runs of the UNMODIFIED
reference on the same inputs (stored by tests/golden/make_golden.py), records compared bit-exactly
after the canonical sort."""
import hashlib
import os
import tempfile

import numpy as np
import pytest

import oracle_lib as ol
from fastga_b200 import formats, lib, synth

pytestmark = pytest.mark.gpu


E2E_PAIRS = {"small_pair": (11, 1_200_000, 3, 0.05, 60_000, 1),
             "scaffolded_15pct": (12, 2_000_000, 6, 0.15, 40_000, 3),
             # no SV breaks: contig-long alignments -> pebble arenas overflow and the retry path runs
             "long_alignments": (13, 6_000_000, 3, 0.03, 0, 1),
             "10mbp": (14, 10_000_000, 5, 0.05, 200_000, 1)}


def _vs_reference(name):
    seed, total, ncontig, div, sv, per_scaffold = E2E_PAIRS[name]
    A, B = synth.make_pair(seed, total, ncontig, div, sv_every=sv)
    with tempfile.TemporaryDirectory() as wd:
        formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", per_scaffold))
        formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", per_scaffold))
        gA = formats.genome_from_fasta(os.path.join(wd, "A.fasta"))
        gB = formats.genome_from_fasta(os.path.join(wd, "B.fasta"))
    ref = ol.reference_run("e2e/" + name)
    st = ref["counters"]
    assert hashlib.md5(gA.bps.tobytes()).hexdigest() == ref["bps_md5_A"]      # the .bps FAtoGDB wrote
    alns, stats = lib.fastga(gA, gB)
    assert stats["nseeds"] == st["seeds"]
    assert stats["nhits"] == st["hits"]
    assert alns.nraw == st["alns"]
    assert len(alns) == st["kept"] == ref["records"]
    mine = alns.canonical_lines()
    assert ol.md5_lines(mine) == ref["aln_md5"]
    return stats


def test_small_pair_bit_exact_vs_reference():
    _vs_reference("small_pair")


def test_scaffolded_15pct_bit_exact_vs_reference():
    _vs_reference("scaffolded_15pct")


def test_long_alignments_exercise_arena_retry():
    _vs_reference("long_alignments")


def test_10mbp_bit_exact_vs_reference():
    _vs_reference("10mbp")


@pytest.mark.parametrize("gap", ["0", "3000", "1000000000"])
def test_hit_groups_any_cut_gives_the_same_records(gap):
    # The extension runs the hits of a band-pair triple as independent groups and re-runs the triple in
    # one piece when a group's alignments reached into the next group (fgb_extend).  Cutting at every
    # hit (0: covered hits are aligned speculatively, found out, re-run), at 3 kbp, or never must all
    # give the records of the default cut.
    A, B = synth.make_pair(21, 3_000_000, 4, 0.08, sv_every=50_000)
    gA, gB = formats.genome_from_arrays(A), formats.genome_from_arrays(B)
    base, st0 = lib.fastga(gA, gB)
    os.environ["FGB_SPEC_GAP"] = gap
    try:
        alns, st1 = lib.fastga(gA, gB)
    finally:
        del os.environ["FGB_SPEC_GAP"]
    assert st1["nhits"] == st0["nhits"] and alns.nraw == base.nraw
    assert ol.md5_lines(alns.canonical_lines()) == ol.md5_lines(base.canonical_lines())


def test_smoke_entry():
    import __graft_entry__
    __graft_entry__.smoke()


EX_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "EXAMPLE")


@pytest.mark.skipif(not os.path.exists(os.path.join(EX_DIR, "HAP1.fasta.gz")),
                    reason="EXAMPLE FASTA not staged under tests/data (data, git-ignored)")
def test_example_hap1_hap2_bit_exact():
    """BASELINE.json configs[0]: EXAMPLE/HAP1 x HAP2 -- 323 569 records, canonical md5 of the
    reference's .1aln (tests/golden/example_golden.json)."""
    import json
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_golden.json")))
    gA = formats.genome_from_fasta(os.path.join(EX_DIR, "HAP1.fasta.gz"))
    gB = formats.genome_from_fasta(os.path.join(EX_DIR, "HAP2.fasta.gz"))
    alns, stats = lib.fastga(gA, gB)
    assert [stats["nkmers1"], stats["nkmers2"]] == gold["kmers"]
    assert stats["nseeds"] == gold["seeds"]
    assert stats["nhits"] == gold["hits"]
    assert alns.nraw == gold["alns"]
    assert len(alns) == gold["kept"]
    assert ol.md5_lines(alns.canonical_lines()) == gold["aln_md5"]


def test_example_regions_wide_band_chunks_bit_exact_vs_oracle():
    """ten 25-40 kbp regions of EXAMPLE (tests/golden/example_regions.npz) whose alignments run
    through bands wider than one 32-lane chunk with the fresh low edge alone in the last chunk: the
    case where the edge must copy the OLD trace-point counter of the diagonal that closed the
    previous chunk (a missing trace point otherwise; found on the full EXAMPLE)"""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_regions.npz"))
    gA = formats.genome_from_arrays([z["a%d" % i] for i in range(10)])
    gB = formats.genome_from_arrays([z["b%d" % i] for i in range(10)])
    want = ol.oracle_pipeline(gA, gB)
    alns, stats = lib.fastga(gA, gB)
    assert stats["nseeds"] == want["nseeds"] and stats["nhits"] == want["nhit"]
    assert alns.canonical_lines() == want["lines"]


def gix_genome():
    A, _ = synth.make_pair(17, 2_500_000, 5, 0.05, sv_every=100_000)
    return A


def test_gix_files_match_reference_gixmake():
    """SURVEY 8 a-4: the .ktab entry stream, the stub index and the part split produced from the
    device table equal what the reference GIXmake writes (equal k-mers canonicalised; stored by
    tests/golden/make_golden.py), and that entry stream imports back into the identical device table."""
    A = gix_genome()
    ref = ol.reference_run("gix/gixmake")
    g = formats.genome_from_arrays(A)
    dg = lib.DeviceGenome(g)
    gx = lib.DeviceGix.build(dg)
    tab, pstart, buck = gx.download()
    assert gx.n == ref["n"]
    pb, cb = formats.gix_bytes(g)
    assert (pb, cb) == (ref["post_bytes"], ref["cont_bytes"]) == (gx.post_bytes, max(gx.cont_bytes, cb))
    index = pstart[1:].astype(np.int64)
    assert hashlib.md5(index.tobytes()).hexdigest() == ref["index_md5"]
    assert list(dg.perm) == ref["perm"][:g.ncontig]
    # part split from the sampler histogram (GIXmake.c:655-691)
    nparts = formats.gix_nparts(g.seqtot, max(g.ncontig, 4), pb, cb, nthreads=4)
    assert nparts == ref["nparts"]
    ks = formats.ksplit_from_buckets(buck, nparts)
    part_first = np.array([int(pstart[k << 14]) for k in ks[:-1]], dtype=np.int64)
    part_n = np.diff(np.concatenate([part_first, [gx.n]]))
    assert list(part_n) == ref["part_n"]
    ent = gx.export_ktab(part_first) if gx.cont_bytes == cb else None
    if ent is None:     # device handle counts real contigs only; re-encode with the padded width
        ent = formats.ktab_entries_from_table(tab, pb, cb, part_first)
    E = 9 + pb + cb
    canon = formats.canonical_ktab(ent, E, index)
    assert hashlib.md5(canon.tobytes()).hexdigest() == ref["entries_md5"]
    # and the reverse direction: the reference's entries (canonical form: the order of equal k-mers
    # differs from the device table's) -> device table
    f = formats.GixFile()
    f.entries, f.n, f.post_bytes, f.cont_bytes, f.index, f.ncontig = canon, gx.n, pb, cb, index, len(ref["perm"])
    imp = lib.DeviceGix.import_ktab(f)
    itab, ipstart, _ = imp.download()
    assert np.array_equal(ipstart, pstart)
    key = lambda t: np.lexsort((t[:, 0] & np.uint64(0xffffffffffff), t[:, 0] >> np.uint64(48), t[:, 1]))
    assert np.array_equal(itab[key(itab)], tab[key(tab)])


# ---------------------------------------------------------------------------------------------
#  edge cases (tests/edge_cases.py): ragged / degenerate inputs, against the reference's runs on
#  them (tests/golden/reference_runs.json)
# ---------------------------------------------------------------------------------------------

import edge_cases  # noqa: E402


@pytest.mark.parametrize("name", sorted(edge_cases.CASES))
def test_edge_case_bit_exact_vs_reference(name):
    A, B, threads, check = edge_cases.CASES[name]()
    ref = ol.reference_run("edge/" + name)
    alns, stats = lib.fastga(formats.genome_from_arrays(A), formats.genome_from_arrays(B))
    assert stats["nseeds"] == ref["counters"].get("seeds", 0)
    lines = alns.canonical_lines()
    assert len(lines) == ref["records"] and ol.md5_lines(lines) == ref["aln_md5"]
    check(alns, stats["nhits"])
