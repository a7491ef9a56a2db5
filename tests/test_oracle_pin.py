"""CPU tests that pin the oracle (oracle/fastga_oracle.c) to the UNMODIFIED reference through
committed golden vectors (tests/golden/reference_golden.json, reference_runs.json and
reference_paths.npz, made by tests/golden/make_golden.py from runs of oracle/_ref): the reference's
counters, its alignment records and its Local_Alignment results on the same seeded inputs."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as ol
from fastga_b200 import formats, synth

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.json")))


def _pair(c):
    A, B = synth.make_pair(c["seed"], c["total"], c["ncontig"], c["div"], sv_every=c["sv"])
    return formats.genome_from_arrays(A), formats.genome_from_arrays(B)


@pytest.mark.parametrize("name", sorted(GOLD))
def test_oracle_reproduces_reference_golden(name):
    g = GOLD[name]
    gA, gB = _pair(g["case"])
    r = ol.oracle_pipeline(gA, gB)
    cnt = g["counters"]
    assert r["nseeds"] == cnt["seeds"]
    assert abs(r["sumlen"] / r["nseeds"] - cnt["avelen"]) < 0.051
    assert r["nhit"] == cnt["hits"]
    assert r["nraw"] == cnt["alns"]
    assert len(r["lines"]) == cnt["kept"] == g["aln_records"]
    assert r["lines"][:3] == g["first_records"]
    assert ol.md5_lines(r["lines"]) == g["aln_md5"]          # bit-exact .1aln content
    for nm, genome, tab, pstart in (("A", gA, r["tabA"], r["pstartA"]), ("B", gB, r["tabB"], r["pstartB"])):
        gg = g["gix"][nm]
        assert hashlib.md5(genome.bps.tobytes()).hexdigest() == gg["bps_md5"]
        assert len(tab) == gg["n"]
        pb, cb = formats.gix_bytes(genome)
        assert (pb, cb) == (gg["post_bytes"], gg["cont_bytes"])
        index = pstart[1:].astype(np.int64)                  # stub index = cumulative counts
        assert hashlib.md5(index.tobytes()).hexdigest() == gg["index_md5"]
        part_first = np.cumsum([0] + gg["part_n"][:-1])
        ent = formats.ktab_entries_from_table(tab, pb, cb, part_first)
        E = 9 + pb + cb                                      # .ktab bytes, equal k-mers canonicalised
        assert hashlib.md5(formats.canonical_ktab(ent, E, index).tobytes()).hexdigest() == gg["entries_md5"]


# ---------------------------------------------------------------------------------------------
#  pins against stored results of oracle/_ref
# ---------------------------------------------------------------------------------------------

class OPath(C.Structure):
    _fields_ = [("abpos", C.c_int), ("bbpos", C.c_int), ("aepos", C.c_int), ("bepos", C.c_int),
                ("diffs", C.c_int), ("tlen", C.c_int), ("trace", C.POINTER(C.c_uint8)), ("tmax", C.c_int)]


def _mutate(rng, a, rate):
    out, i = [], 0
    r = rng.random(len(a) * 2 + 8)
    q = 0
    while i < len(a):
        u = r[q]
        q += 1
        if u < rate * 0.8:
            out.append((a[i] + rng.integers(1, 4)) % 4)
            i += 1
        elif u < rate * 0.9:
            out.append(rng.integers(0, 4))
        elif u < rate:
            i += 1
        else:
            out.append(a[i])
            i += 1
    return np.array(out, dtype=np.int8)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_local_alignment_bit_exact_vs_reference_library(seed):
    _la_compare(seed, borders=False)


@pytest.mark.parametrize("seed", [11, 12])
def test_local_alignment_with_band_borders_vs_reference_library(seed):
    """lbord / hbord >= 0 confine the band to [low-lbord, hgh+hbord] (align.c:1466-1481): what
    align_contigs passes for a contig against itself (FastGA.c:3247-3262); the CUDA waves take the
    same minp/maxp arguments but FastGA's non-self mode never sets them"""
    _la_compare(seed, borders=True)


def la_calls(seed, borders):
    """400 Local_Alignment calls on random sequence pairs: (a, b, acomp, low, hgh, anti, lbord, hbord)"""
    rng = np.random.default_rng(seed)
    for _ in range(400):
        L = int(rng.integers(300, 5000))
        rate = float(rng.choice([0.0, 0.02, 0.05, 0.1, 0.15, 0.3]))
        core = rng.integers(0, 4, L).astype(np.int8)
        fa, fb, ta, tb = (rng.integers(0, 4, int(rng.integers(0, 400))).astype(np.int8) for _ in range(4))
        if rng.random() < 0.3:
            fa = fa[:0]
        if rng.random() < 0.3:
            tb = tb[:0]
        a = np.concatenate([fa, core, ta])
        b = np.concatenate([fb, _mutate(rng, core, rate), tb])
        acomp = int(rng.random() < 0.5)
        xa, xb = len(fa) + L // 2, len(fb) + L // 2
        d, anti = xa - xb, xa + xb + int(rng.integers(-100, 100))
        low, hgh = d - int(rng.integers(0, 80)), d + int(rng.integers(0, 80))
        lb = hb = -1
        if borders:
            lb = int(rng.integers(0, 40)) if rng.random() < 0.7 else -1
            hb = int(rng.integers(0, 40)) if rng.random() < 0.7 else -1
        yield a, b, acomp, low, hgh, anti, lb, hb


def _la_compare(seed, borders):
    """the oracle's Local_Alignment against the reference's on the calls of la_calls"""
    orc = ol.orc()
    orc.orc_local_alignment.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + \
        [C.c_int] * 6 + [C.POINTER(OPath)]
    ospec, _tabs, _ = ol.make_spec(np.array([.25] * 4, np.float32), 0.7)
    owork = C.c_void_p(orc.orc_new_work())
    want, wtrace = ol.reference_paths("la_%s%d" % ("b" if borders else "", seed))
    for it, (a, b, acomp, low, hgh, anti, lb, hb) in enumerate(la_calls(seed, borders)):
        ab, bb = ol._framed(a), ol._framed(b)
        op = OPath()
        orc.orc_local_alignment(owork, C.byref(ospec), ab.ctypes.data + 1, len(a), bb.ctypes.data + 1, len(b),
                                acomp, low, hgh, anti, lb, hb, C.byref(op))
        ot = np.ctypeslib.as_array(op.trace, shape=(max(op.tlen, 1),))[:op.tlen] if op.tlen else np.zeros(0, np.uint8)
        assert tuple(int(v) for v in want[it]) == \
               (op.abpos, op.bbpos, op.aepos, op.bepos, op.diffs, op.tlen), (it, len(a), acomp, lb, hb)
        assert np.array_equal(wtrace[it], ot), (it, len(a), acomp, lb, hb)
    assert it + 1 == len(want)


def test_oracle_vs_live_reference_run(tmp_path):
    """the oracle against a reference run on a scaffolded pair (tests/golden/reference_runs.json),
    and the product's FASTA reader against the contig split of the reference's FAtoGDB"""
    A, B = synth.make_pair(31, 600_000, 3, 0.07, sv_every=30_000)
    wd = str(tmp_path)
    formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", 1))
    formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", 3))
    ref = ol.reference_run("oracle/scaffolded")
    st = ref["counters"]
    gA = formats.genome_from_fasta(os.path.join(wd, "A.fasta"))
    gB = formats.genome_from_fasta(os.path.join(wd, "B.fasta"))
    gdb = ref["gdb_B"]
    assert list(gB.clen) == gdb["clen"] and list(gB.sbeg) == gdb["sbeg"] and list(gB.scaf) == gdb["scaf"]
    r = ol.oracle_pipeline(gA, gB)
    assert (r["nseeds"], r["nhit"], r["nraw"], len(r["lines"])) == (st["seeds"], st["hits"], st["alns"], st["kept"])
    assert len(r["lines"]) == ref["records"] and ol.md5_lines(r["lines"]) == ref["aln_md5"]


def test_written_1aln_is_read_by_reference_tools(tmp_path):
    """SURVEY 8 a-16: a .1aln written by formats.write_1aln_ascii carries the records of the
    reference's own .1aln, in the text ONEview reads back (tests/golden/reference_runs.json).  Where
    the reference tools are built, the file also goes through them: ONEview returns the same records
    and -- after ONEview -b adds the binary index the threaded readers need -- ALNtoPAF, next to the
    reference-made GDBs, gives the same PAF as from the reference's own .1aln."""
    A, B = synth.make_pair(41, 500_000, 3, 0.06, sv_every=40_000)
    wd = str(tmp_path)
    formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", 2))
    formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", 1))
    gA = formats.genome_from_fasta(os.path.join(wd, "A.fasta"))
    gB = formats.genome_from_fasta(os.path.join(wd, "B.fasta"))
    r = ol.oracle_pipeline(gA, gB)
    formats.write_1aln_ascii(os.path.join(wd, "mine.1aln"), r["alns"], gA, gB, "./A.1gdb", "./B.1gdb", wd)
    ref = ol.reference_run("oracle/written_1aln")
    with open(os.path.join(wd, "mine.1aln")) as f:
        mine = ol.records_from_text(f.read())
    assert len(mine) == ref["records"] and ol.md5_lines(mine) == ref["aln_md5"]
    if not ol.have_ref():
        return
    ol.ref_fastga(wd, "A", "B", threads=4)
    assert ol.oneview_records(os.path.join(wd, "mine.1aln")) == ol.oneview_records(os.path.join(wd, "ref.1aln"))
    paf_ref = sorted(ol.run_ref(["ALNtoPAF", "-T2", "ref"], cwd=wd).split("\n"))
    # the threaded converters need ONEcode's binary index: ONEview -b turns the ASCII file into it
    ol.run_ref(["ONEview", "-b", "-o", "mineb.1aln", "mine.1aln"], cwd=wd)
    paf_mine = sorted(ol.run_ref(["ALNtoPAF", "-T2", "mineb"], cwd=wd).split("\n"))
    assert len(paf_ref) > 3 and paf_mine == paf_ref


def _assert_reference_run(r, key):
    ref = ol.reference_run(key)
    assert r["nseeds"] == ref["counters"].get("seeds", 0)
    assert len(r["lines"]) == ref["records"] and ol.md5_lines(r["lines"]) == ref["aln_md5"]


import edge_cases  # noqa: E402


@pytest.mark.parametrize("name", sorted(edge_cases.CASES))
def test_oracle_edge_cases_vs_live_reference(name):
    """the oracle on the edge-case inputs of tests/edge_cases.py, against the reference's run on them"""
    A, B, threads, check = edge_cases.CASES[name]()
    r = ol.oracle_pipeline(formats.genome_from_arrays(A), formats.genome_from_arrays(B))
    _assert_reference_run(r, "edge/" + name)
    check(r["alns"], r["nhit"])


def example_regions():
    z = np.load(os.path.join(ol.GOLDEN, "example_regions.npz"))
    return [z["a%d" % i] for i in range(10)], [z["b%d" % i] for i in range(10)]


def test_oracle_on_example_regions_vs_live_reference():
    """the EXAMPLE regions fixture of the GPU regression test, oracle against the reference's run on it"""
    A, B = example_regions()
    r = ol.oracle_pipeline(formats.genome_from_arrays(A), formats.genome_from_arrays(B))
    _assert_reference_run(r, "oracle/example_regions")


def _self_genomes():
    """genomes with internal homology for SELF mode (FastGA A): a diverged duplication inside and
    across contigs plus an inverted copy, and two tandem-repeat genomes (near-diagonal chains: the
    'nothing across the main diagonal' branch and the band borders of align_contigs)"""
    rng = np.random.default_rng(5)
    a = rng.integers(0, 4, 300_000, dtype=np.uint8)
    dup = synth.diverged_copy(rng, a[50_000:150_000], 0.05, sv_every=40_000)
    c0 = np.concatenate([a, dup, rng.integers(0, 4, 20_000, dtype=np.uint8)])
    c1 = np.concatenate([rng.integers(0, 4, 100_000, dtype=np.uint8),
                         synth.diverged_copy(rng, a[200_000:280_000], 0.04, sv_every=30_000),
                         (3 - a[10_000:60_000][::-1]).astype(np.uint8)])
    out = {"dup": [c0, c1[:len(c1) - 3]]}
    for seed in (61, 62):
        rng = np.random.default_rng(seed)
        parts = []
        while sum(len(p) for p in parts) < 500_000:
            parts.append(rng.integers(0, 4, int(rng.integers(20_000, 60_000)), dtype=np.uint8))
            unit = rng.integers(0, 4, int(rng.integers(150, 1200)), dtype=np.uint8)
            parts.append(np.concatenate([synth._small_mutations(rng, unit, 0.03)
                                         for _ in range(int(rng.integers(8, 60)))]))
        g = np.concatenate(parts)[:500_000]
        cut = int(rng.integers(200_000, 300_000))
        out["tandem%d" % seed] = [g[:cut], g[cut:]]
    # C-strand self pairs, identical contigs, a palindrome, a long near-diagonal repeat array
    rng = np.random.default_rng(101)
    a = rng.integers(0, 4, 200_000, dtype=np.uint8)
    inv = (3 - a[30_000:90_000][::-1]).astype(np.uint8)
    out["inverted_dup"] = [np.concatenate([a, rng.integers(0, 4, 5000, dtype=np.uint8),
                                           synth._small_mutations(rng, inv, 0.03)])]
    out["identical_contigs"] = [a.copy(), a.copy()[:199_990], rng.integers(0, 4, 50_000, dtype=np.uint8)]
    out["palindrome"] = [np.concatenate([a[:60_000], (3 - a[:60_000][::-1]).astype(np.uint8)]),
                         rng.integers(0, 4, 30_001, dtype=np.uint8)]
    rng = np.random.default_rng(102)
    unit = rng.integers(0, 4, 5000, dtype=np.uint8)
    out["near_diagonal_repeats"] = [np.concatenate(
        [rng.integers(0, 4, 50_000, dtype=np.uint8)] +
        [synth._small_mutations(rng, unit, 0.04) for _ in range(30)] +
        [rng.integers(0, 4, 50_000, dtype=np.uint8)])]
    return out


@pytest.mark.parametrize("name", ["dup", "tandem61", "tandem62", "inverted_dup", "identical_contigs",
                                  "palindrome", "near_diagonal_repeats"])
def test_oracle_self_mode_vs_live_reference(name):
    """SURVEY row a-7 groundwork: the oracle's SELF mode (self block rule, band borders for a contig
    against itself) against `FastGA A` of the reference (tests/golden/reference_runs.json)"""
    G = _self_genomes()[name]
    ref = ol.reference_run("self/" + name)
    st = ref["counters"]
    r = ol.oracle_pipeline_self(formats.genome_from_arrays(G))
    # every thread of the reference halves its own pair count (FastGA.c:1907): off by < #threads
    assert abs(r["nseeds"] // 2 - st["seeds"]) < 4
    assert r["nhit"] == st["hits"] and r["nraw"] == st["alns"]
    assert len(r["lines"]) == ref["records"] and ol.md5_lines(r["lines"]) == ref["aln_md5"]
