"""Regenerates the golden files of tests/golden by running the UNMODIFIED reference (oracle/_ref,
which build() compiles where the reference sources are present).  Committed with its output.

reference_golden.json: for each case a synthetic pair from fastga_b200.synth (pure function of the
seed), the reference's own -v counters (seeds / hits / aln's / non-redundant), the md5 of the
canonical-sorted ONEview dump of its .1aln, and the md5s of its GIX files' content (entries +
index), so that the oracle -- and through it the CUDA path -- can be pinned without the reference.

reference_runs.json: what the reference produced on the inputs of the tests that compare with it
(FastGA runs, a GIXmake run, the msd_sort / rmsd_sort seams, Compute_Trace_PTS scripts), keyed as
the tests look them up.

reference_paths.npz: the reference's Local_Alignment results on the call lists of the Local_Alignment
tests: <key>_paths (n, 6) int32 rows abpos bbpos aepos bepos diffs tlen, <key>_traces the trace
bytes of all calls concatenated.
"""
import ctypes as C
import hashlib
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np          # noqa: E402
import oracle_lib as ol     # noqa: E402
from fastga_b200 import formats, synth   # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = {
    "pair_a": dict(seed=21, total=300_000, ncontig=2, div=0.05, sv=40_000, per_scaffold=1),
    "pair_b": dict(seed=22, total=800_000, ncontig=4, div=0.10, sv=50_000, per_scaffold=2),
    "pair_c": dict(seed=23, total=500_000, ncontig=3, div=0.02, sv=0, per_scaffold=1),
}


def reference_golden():
    out = {}
    for name, c in CASES.items():
        A, B = synth.make_pair(c["seed"], c["total"], c["ncontig"], c["div"], sv_every=c["sv"])
        with tempfile.TemporaryDirectory() as wd:
            formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", c["per_scaffold"]))
            formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", c["per_scaffold"]))
            log = ol.ref_fastga(wd, "A", "B", threads=4)
            st = ol.parse_fastga_log(log)
            recs = ol.oneview_records(os.path.join(wd, "ref.1aln"))
            g = {}
            for nm in ("A", "B"):
                gx = formats.read_gix(os.path.join(wd, nm + ".gix"))
                g[nm] = {"n": gx.n, "post_bytes": gx.post_bytes, "cont_bytes": gx.cont_bytes,
                         "nparts": gx.nparts, "part_n": [int(x) for x in gx.part_n],
                         "entries_md5": hashlib.md5(formats.canonical_ktab(gx.entries, gx.esize, gx.index).tobytes()).hexdigest(),
                         "index_md5": hashlib.md5(gx.index.tobytes()).hexdigest(),
                         "bps_md5": hashlib.md5(open(os.path.join(wd, "." + nm + ".bps"), "rb").read()).hexdigest()}
        out[name] = {"case": c, "counters": st, "aln_md5": ol.md5_lines(recs), "aln_records": len(recs),
                     "first_records": recs[:3], "gix": g}
        print(name, st, len(recs))
    with open(os.path.join(HERE, "reference_golden.json"), "w") as f:
        json.dump(out, f, indent=1)


# ---------------------------------------------------------------------------------------------
#  libfastga_ref.so: the reference's align.h entry points
# ---------------------------------------------------------------------------------------------

class Path(C.Structure):
    _fields_ = [("trace", C.c_void_p), ("tlen", C.c_int), ("diffs", C.c_int), ("abpos", C.c_int),
                ("bbpos", C.c_int), ("aepos", C.c_int), ("bepos", C.c_int)]


class Alignment(C.Structure):
    _fields_ = [("path", C.POINTER(Path)), ("flags", C.c_uint32), ("aseq", C.c_void_p), ("bseq", C.c_void_p),
                ("alen", C.c_int), ("blen", C.c_int)]


def _ref_lib():
    ref = C.CDLL(ol.REF_SO)
    ref.New_Work_Data.restype = C.c_void_p
    ref.New_Align_Spec.restype = C.c_void_p
    ref.New_Align_Spec.argtypes = [C.c_double, C.c_int, C.POINTER(C.c_float), C.c_int]
    ref.Local_Alignment.argtypes = [C.POINTER(Alignment), C.c_void_p, C.c_void_p] + [C.c_int] * 5
    ref.Compute_Trace_PTS.argtypes = [C.POINTER(Alignment), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    return ref


def local_alignments(calls, freq):
    """Local_Alignment(aln, work, spec(0.7, 100, freq), low, hgh, anti, lbord, hbord) on each call
    (a, b, comp, low, hgh, anti, lbord, hbord) -> (paths, traces) as stored in reference_paths.npz"""
    ref = _ref_lib()
    work = ref.New_Work_Data()
    spec = ref.New_Align_Spec(0.7, 100, (C.c_float * 4)(*[float(v) for v in freq]), 0)
    paths, traces = [], []
    for a, b, comp, low, hgh, anti, lb, hb in calls:
        fa, fb = ol._framed(a), ol._framed(b)
        p = Path()
        al = Alignment(C.pointer(p), 2 if comp else 0, fa.ctypes.data + 1, fb.ctypes.data + 1, len(a), len(b))
        assert ref.Local_Alignment(C.byref(al), work, spec, low, hgh, anti, lb, hb) == 0
        rt = np.ctypeslib.as_array(C.cast(p.trace, C.POINTER(C.c_uint16)), shape=(max(p.tlen, 1),))[:p.tlen]
        paths.append((p.abpos, p.bbpos, p.aepos, p.bepos, p.diffs, p.tlen))
        traces.append(rt.astype(np.uint8))
    return np.array(paths, dtype=np.int32), np.concatenate(traces)


def trace_scripts(gA, gB, alns):
    """Compute_Trace_PTS(aln, work, 100, GREEDIEST, 1, -1) as ALNtoPAF.c:251-272 calls it, per
    alignment: [comp aread bread abpos bbpos aepos bepos, diffs, script length, script md5]"""
    ref = _ref_lib()
    work = ref.New_Work_Data()
    A = [ol._framed(gA.contig(c)) for c in range(gA.ncontig)]
    B = [ol._framed(gB.contig(c)) for c in range(gB.ncontig)]
    BC = [ol._framed(3 - gB.contig(c)[::-1]) for c in range(gB.ncontig)]
    out = []
    for i in range(len(alns)):
        comp, ar, br, ab, bb, ae, be, df, tl = (int(x) for x in alns.fields[i])
        pts = alns.trace(i).astype(np.uint16)            # Decompress_TraceTo16
        p = Path(pts.ctypes.data, tl, df, ab, bb, ae, be)
        a, b = A[ar], (BC[br] if comp else B[br])
        al = Alignment(C.pointer(p), 2 if comp else 0, a.ctypes.data + 1, b.ctypes.data + 1, len(a) - 2, len(b) - 2)
        assert ref.Compute_Trace_PTS(C.byref(al), work, 100, 0, 1, -1) == 0
        sc = np.ctypeslib.as_array(C.cast(p.trace, C.POINTER(C.c_int32)), shape=(max(p.tlen, 1),))[:p.tlen]
        sc = np.ascontiguousarray(sc, dtype=np.int32)
        out.append([comp, ar, br, ab, bb, ae, be, int(p.diffs), len(sc), hashlib.md5(sc.tobytes()).hexdigest()])
    assert len({tuple(r[:7]) for r in out}) == len(out)
    return out


# ---------------------------------------------------------------------------------------------
#  reference runs on the test inputs
# ---------------------------------------------------------------------------------------------

def fastga_run(A, B, threads, a_scaf=1, b_scaf=1, gdb_B=False):
    """FastGA -v -k -T<threads> on FASTA files of the contigs (B None: SELF mode)"""
    with tempfile.TemporaryDirectory() as wd:
        formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", a_scaf))
        if B is not None:
            formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", b_scaf))
        st = ol.parse_fastga_log(ol.ref_fastga(wd, "A", "B" if B is not None else None, threads=threads))
        recs = ol.oneview_records(os.path.join(wd, "ref.1aln"))
        out = {"counters": st, "records": len(recs), "aln_md5": ol.md5_lines(recs),
               "bps_md5_A": hashlib.md5(open(os.path.join(wd, ".A.bps"), "rb").read()).hexdigest()}
        if gdb_B:
            clen, _, scaf, sbeg = ol.read_gdb_ascii(os.path.join(wd, "B.1gdb"))
            out["gdb_B"] = {"clen": clen.tolist(), "scaf": scaf.tolist(), "sbeg": sbeg.tolist()}
    return out


def written_1aln_run():
    """the reference's records for the .1aln writer test, after checking that the ASCII .1aln the
    writer makes reads back through ONEview as the same records as its own text"""
    A, B = synth.make_pair(41, 500_000, 3, 0.06, sv_every=40_000)
    out = fastga_run(A, B, 4, a_scaf=2)
    with tempfile.TemporaryDirectory() as wd:
        formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", 2))
        formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", 1))
        gA = formats.genome_from_fasta(os.path.join(wd, "A.fasta"))
        gB = formats.genome_from_fasta(os.path.join(wd, "B.fasta"))
        r = ol.oracle_pipeline(gA, gB)
        path = os.path.join(wd, "mine.1aln")
        formats.write_1aln_ascii(path, r["alns"], gA, gB, "./A.1gdb", "./B.1gdb", wd)
        with open(path) as f:
            assert ol.records_from_text(f.read()) == ol.oneview_records(path)
    return out


def gix_run(A):
    with tempfile.TemporaryDirectory() as wd:
        formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", 2))
        ol.run_ref(["GIXmake", "-T4", "-P" + wd, "A"], cwd=wd)
        ref = formats.read_gix(os.path.join(wd, "A.gix"))
    return {"n": ref.n, "post_bytes": ref.post_bytes, "cont_bytes": ref.cont_bytes,
            "index_md5": hashlib.md5(ref.index.tobytes()).hexdigest(), "perm": ref.perm.tolist(),
            "nparts": ref.nparts, "part_n": [int(x) for x in ref.part_n],
            "entries_md5": hashlib.md5(formats.canonical_ktab(ref.entries, ref.esize, ref.index).tobytes()).hexdigest()}


def sort_seams():
    import test_gpu_stages as ts
    ref = C.CDLL(ol.REF_SO)
    ref.msd_sort.argtypes = ts.MSD_ARGTYPES
    ref.rmsd_sort.argtypes = ts.RMSD_ARGTYPES
    a, n, rsize, ksize, part, beg, end = ts.msd_input()
    ref.msd_sort(a.ctypes.data, n, rsize, ksize, part.ctypes.data, beg, end, 4)
    r = a[:n * rsize].reshape(n, rsize)
    msd = {"sentinel": int(a[n * rsize]), "keys_md5": hashlib.md5(np.ascontiguousarray(r[:, :ksize]).tobytes()).hexdigest(),
           "payload_md5": ts.msd_payload_md5(r, ksize)}
    a, n, rsize, nparts, part, nthreads = ts.rmsd_input()
    p = (ts._Range * nthreads)()
    n1 = ref.rmsd_sort(a.ctypes.data, n, rsize, rsize, nparts, part.ctypes.data, nthreads, p)
    rmsd = {"ranges": [[p[i].beg, p[i].end, p[i].off] for i in range(n1)], "md5": hashlib.md5(a.tobytes()).hexdigest()}
    return msd, rmsd


def reference_runs():
    import edge_cases
    import test_gpu_e2e as te
    import test_gpu_trace as tt
    import test_oracle_pin as tp
    out = {}
    A, B = synth.make_pair(31, 600_000, 3, 0.07, sv_every=30_000)
    out["oracle/scaffolded"] = fastga_run(A, B, 4, b_scaf=3, gdb_B=True)
    out["oracle/written_1aln"] = written_1aln_run()
    out["oracle/example_regions"] = fastga_run(*tp.example_regions(), 4)
    for name, case in sorted(edge_cases.CASES.items()):
        A, B, threads, _ = case()
        out["edge/" + name] = fastga_run(A, B, threads)
    for name, G in tp._self_genomes().items():
        out["self/" + name] = fastga_run(G, None, 4)
    for name, (seed, total, ncontig, div, sv, per_scaffold) in te.E2E_PAIRS.items():
        A, B = synth.make_pair(seed, total, ncontig, div, sv_every=sv)
        out["e2e/" + name] = fastga_run(A, B, 8, a_scaf=per_scaffold, b_scaf=per_scaffold)
    out["gix/gixmake"] = gix_run(te.gix_genome())
    for name, args in tt.TRACE_PAIRS.items():
        gA, gB = tt.trace_pair(*args)
        out["trace/" + name] = {"scripts": trace_scripts(gA, gB, ol.oracle_pipeline(gA, gB)["alns"])}
    out["seam/msd_sort"], out["seam/rmsd_sort"] = sort_seams()
    for k, v in out.items():
        print(k, v.get("counters"), v.get("records"))
    with open(os.path.join(HERE, "reference_runs.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)


def reference_paths():
    import test_gpu_align_seam as tg
    import test_oracle_pin as tp
    arrays = {}
    for seed, borders in ((1, False), (2, False), (3, False), (11, True), (12, True)):
        key = "la_%s%d" % ("b" if borders else "", seed)
        arrays[key + "_paths"], arrays[key + "_traces"] = local_alignments(tp.la_calls(seed, borders), [.25] * 4)
    for borders in (False, True):
        A, B, jobs = tg.seam_jobs(borders)
        calls = [((3 - A[i][::-1]).astype(np.uint8) if comp else A[i], B[j], comp, low, hgh, anti, lb, hb)
                 for i, j, comp, low, hgh, anti, lb, hb in jobs.tolist()]
        key = "seam_%s" % borders
        arrays[key + "_paths"], arrays[key + "_traces"] = \
            local_alignments(calls, formats.genome_from_arrays(A).freq)
    np.savez_compressed(os.path.join(HERE, "reference_paths.npz"), **arrays)


def main():
    if not ol.have_ref():
        sys.exit("oracle/_ref has not been built: build() makes it where the reference sources are present")
    which = sys.argv[1:] or ["golden", "runs", "paths"]
    if "golden" in which:
        reference_golden()
    if "paths" in which:
        reference_paths()
    if "runs" in which:
        reference_runs()


if __name__ == "__main__":
    main()
