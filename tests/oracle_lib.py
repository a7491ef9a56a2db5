"""TEST INFRASTRUCTURE: ctypes access to oracle/liboracle.so (the CPU restatement) and to the
unmodified reference built into oracle/_ref (binaries + libfastga_ref.so)."""
import ctypes as C
import hashlib
import json
import os
import re
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF_SO = os.path.join(REF_DIR, "libfastga_ref.so")

_orc = None


GOLDEN = os.path.join(ROOT, "tests", "golden")
_runs = None


def have_ref():
    return os.path.exists(os.path.join(REF_DIR, "FastGA")) and os.path.exists(REF_SO)


def reference_run(key):
    """What the unmodified reference produced for one test input, as stored in
    tests/golden/reference_runs.json by tests/golden/make_golden.py."""
    global _runs
    if _runs is None:
        with open(os.path.join(GOLDEN, "reference_runs.json")) as f:
            _runs = json.load(f)
    return _runs[key]


def reference_paths(key):
    """The reference's Local_Alignment results for one list of calls (tests/golden/reference_paths.npz):
    (n, 6) int32 rows abpos bbpos aepos bepos diffs tlen, and the traces of all calls concatenated."""
    with np.load(os.path.join(GOLDEN, "reference_paths.npz")) as z:
        paths, traces = z[key + "_paths"], z[key + "_traces"]
    toff = np.concatenate([[0], np.cumsum(paths[:, 5].astype(np.int64))])
    return paths, [traces[toff[i]:toff[i + 1]] for i in range(len(paths))]


def orc():
    global _orc
    if _orc is None:
        if not os.path.exists(ORACLE_SO):
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", ORACLE_SO,
                                   os.path.join(ROOT, "oracle", "fastga_oracle.c")])
        _orc = C.CDLL(ORACLE_SO)
        _orc.orc_gix_build.restype = C.c_int64
        _orc.orc_merge.restype = C.c_int64
        _orc.orc_syncmers.restype = C.c_int64
        _orc.orc_new_work.restype = C.c_void_p
        if hasattr(_orc, "orc_search"):
            _orc.orc_search.restype = C.c_int64
    return _orc


class OrcSeed(C.Structure):
    _fields_ = [("plen", C.c_uint8), ("comp", C.c_uint8), ("icont", C.c_uint16), ("jcont", C.c_uint16),
                ("ipost", C.c_uint32), ("jpost", C.c_uint32)]


SEED_DT = np.dtype([("plen", "u1"), ("comp", "u1"), ("icont", "u2"), ("jcont", "u2"),
                    ("ipost", "u4"), ("jpost", "u4")], align=True)


class OrcLayout(C.Structure):
    _fields_ = [("anti_bits", C.c_int), ("band_bits", C.c_int), ("jc_bits", C.c_int), ("ic_bits", C.c_int),
                ("amxpos", C.c_int64), ("bmxpos", C.c_int64)]


def contig_rank(clen):
    """rank of each contig in the decreasing-length order; lengths must be pairwise distinct so
    the libc qsort tie order (GIXmake.c:1959) cannot matter"""
    clen = np.asarray(clen)
    perm = np.argsort(-clen, kind="stable").astype(np.int32)
    rank = np.empty_like(perm)
    rank[perm] = np.arange(len(clen), dtype=np.int32)
    return perm, rank


def gix_build(genome, crank):
    """oracle table of a formats.Genome: (n,2) uint64 records [lo,hi] + pstart"""
    o = orc()
    nc = genome.ncontig
    seqs = [np.ascontiguousarray(genome.contig(c)) for c in range(nc)]
    arr = (C.c_void_p * nc)(*[s.ctypes.data for s in seqs])
    tab = C.c_void_p()
    pstart = np.zeros((1 << 24) + 1, dtype=np.uint32)
    crank = np.ascontiguousarray(crank, dtype=np.int32)
    n = o.orc_gix_build(nc, arr, genome.clen.ctypes.data_as(C.c_void_p), crank.ctypes.data_as(C.c_void_p),
                        C.byref(tab), pstart.ctypes.data_as(C.c_void_p))
    out = np.ctypeslib.as_array(C.cast(tab, C.POINTER(C.c_uint64)), shape=(max(n, 1), 2))[:n].copy()
    o.orc_free(tab)
    return out, pstart


def merge(T1, T2, pstart2, freq=10):
    o = orc()
    T1 = np.ascontiguousarray(T1, dtype=np.uint64)
    T2 = np.ascontiguousarray(T2, dtype=np.uint64)
    sl = C.c_int64()
    args = [T1.ctypes.data_as(C.c_void_p), C.c_int64(len(T1)), T2.ctypes.data_as(C.c_void_p),
            C.c_int64(len(T2)), pstart2.ctypes.data_as(C.c_void_p), C.c_int(freq)]
    n = o.orc_merge(*args, None, C.byref(sl))
    seeds = np.zeros(n, dtype=SEED_DT)
    o.orc_merge(*args, seeds.ctypes.data_as(C.c_void_p), C.byref(sl))
    return seeds, sl.value


def self_merge(T, pstart, freq=10):
    """SELF mode (FastGA A): every entry of the one table against its own block (orc_self_merge)"""
    o = orc()
    T = np.ascontiguousarray(T, dtype=np.uint64)
    sl = C.c_int64()
    args = [T.ctypes.data_as(C.c_void_p), C.c_int64(len(T)), pstart.ctypes.data_as(C.c_void_p), C.c_int(freq)]
    o.orc_self_merge.restype = C.c_int64
    n = o.orc_self_merge(*args, None, C.byref(sl))
    seeds = np.zeros(n, dtype=SEED_DT)
    o.orc_self_merge(*args, seeds.ctypes.data_as(C.c_void_p), C.byref(sl))
    return seeds, sl.value


def seed_records(seeds, layout, sort=True):
    o = orc()
    out = np.zeros((len(seeds), 2), dtype=np.uint64)
    L = OrcLayout(*layout)
    o.orc_seed_records(seeds.ctypes.data_as(C.c_void_p), C.c_int64(len(seeds)), C.byref(L),
                       out.ctypes.data_as(C.c_void_p), C.c_int(1 if sort else 0))
    return out


# ------------------------------------------------------------------------------------------
#  the unmodified reference
# ------------------------------------------------------------------------------------------

def ref_env():
    env = dict(os.environ)
    env["PATH"] = REF_DIR + os.pathsep + env.get("PATH", "")
    return env


def run_ref(args, cwd, timeout=3600):
    r = subprocess.run(args, cwd=cwd, env=ref_env(), stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference command failed: %s\n%s" % (" ".join(args), r.stdout[-2000:]))
    return r.stdout


def ref_fastga(workdir, a, b, out="ref", threads=8, extra=()):
    """FastGA -v -k -T<n> -1:<out> a [b] in workdir (b None: SELF mode); returns the -v log"""
    return run_ref(["FastGA", "-v", "-k", "-T%d" % threads, "-P" + workdir, "-1:" + out] + list(extra) +
                   ([a, b] if b is not None else [a]), cwd=workdir)


def parse_fastga_log(log):
    log = log.replace("\r", "\n")
    d = {}
    m = re.search(r"Total seeds = ([\d,]+), ave\. len = ([\d.]+)", log)
    if m:
        d["seeds"] = int(m.group(1).replace(",", ""))
        d["avelen"] = float(m.group(2))
    m = re.search(r"Total hits over \d+bp = (\d+), (\d+) aln's, (\d+) non-redundant", log)
    if m:
        d["hits"], d["alns"], d["kept"] = int(m.group(1)), int(m.group(2)), int(m.group(3))
    return d


def oneview_records(path):
    """Canonical form of a .1aln: one text line per alignment ('A ..| R | D ..| T ..| X ..'),
    sorted (SURVEY 8c)."""
    out = subprocess.run([os.path.join(REF_DIR, "ONEview"), path], stdout=subprocess.PIPE, text=True,
                         check=True).stdout
    return records_from_text(out)


def records_from_text(out):
    """canonical records of ONEcode ASCII text: ONEview's dump, or an ASCII .1aln as it is"""
    recs, cur = [], None
    for line in out.split("\n"):
        if line.startswith("A "):
            if cur is not None:
                recs.append(cur)
            cur = line
        elif cur is not None and line[:2] in ("R", "R ", "D ", "T ", "X "):
            cur += " | " + line
        elif cur is not None and line.startswith("R"):
            cur += " | " + line
    if cur is not None:
        recs.append(cur)
    recs.sort()
    return recs


def md5_lines(lines):
    h = hashlib.md5()
    for l in lines:
        h.update(l.encode() + b"\n")
    return h.hexdigest()


def read_gdb_ascii(path):
    """contig lengths, scaffold names etc. of a .1gdb through ONEview"""
    out = subprocess.run([os.path.join(REF_DIR, "ONEview"), path], stdout=subprocess.PIPE, text=True,
                         check=True).stdout
    clen, names, scaf, sbeg = [], [], [], []
    pos = 0
    for line in out.split("\n"):
        if line.startswith("S "):
            names.append(line.split(" ", 2)[2])
            pos = 0
        elif line.startswith("G "):
            pos += int(line.split()[1])
        elif line.startswith("C "):
            n = int(line.split()[1])
            clen.append(n)
            scaf.append(len(names) - 1)
            sbeg.append(pos)
            pos += n
    return np.array(clen, np.int64), names, np.array(scaf, np.int32), np.array(sbeg, np.int64)


# ------------------------------------------------------------------------------------------
#  chain scan + extension through the oracle
# ------------------------------------------------------------------------------------------

class OrcSpec(C.Structure):
    _fields_ = [("tspace", C.c_int), ("path_ave", C.c_int), ("score", C.POINTER(C.c_int16)),
                ("table", C.POINTER(C.c_int16))]


class OrcParams(C.Structure):
    _fields_ = [("chain_break", C.c_int), ("chain_min", C.c_int), ("align_min", C.c_int),
                ("align_rate", C.c_double)]


OVL_DT = np.dtype([("comp", "i4"), ("aread", "i4"), ("bread", "i4"), ("abpos", "i4"), ("bbpos", "i4"),
                   ("aepos", "i4"), ("bepos", "i4"), ("diffs", "i4"), ("tlen", "i4"), ("toff", "i8")],
                  align=True)


def make_spec(freq, ave_corr=0.7, tspace=100):
    o = orc()
    tabs = np.zeros(65536, dtype=np.int16)
    ave = C.c_int()
    f = np.ascontiguousarray(freq, dtype=np.float32)
    o.orc_align_spec(C.c_double(ave_corr), f.ctypes.data_as(C.c_void_p), tabs.ctypes.data_as(C.c_void_p),
                     C.byref(ave))
    spec = OrcSpec(tspace, ave.value, C.cast(tabs.ctypes.data, C.POINTER(C.c_int16)),
                   C.cast(tabs.ctypes.data + 65536, C.POINTER(C.c_int16)))
    return spec, tabs, ave.value


def _framed(a):
    b = np.empty(len(a) + 2, dtype=np.int8)
    b[0] = 4
    b[-1] = 4
    b[1:-1] = a
    return b


def search(recs, layout, gA, gB, perm1, perm2, freq, chain_break=2000, chain_min=170, align_min=100,
           align_rate=0.3):
    """oracle alignments in reference discovery order: (records, trace pool, nhit)"""
    o = orc()
    spec, tabs, _ = make_spec(freq, 1.0 - align_rate)
    A = [_framed(gA.contig(c)) for c in range(gA.ncontig)]
    AC = [_framed(3 - gA.contig(c)[::-1]) for c in range(gA.ncontig)]
    B = [_framed(gB.contig(c)) for c in range(gB.ncontig)]
    pa = (C.c_void_p * gA.ncontig)(*[x.ctypes.data + 1 for x in A])
    pac = (C.c_void_p * gA.ncontig)(*[x.ctypes.data + 1 for x in AC])
    pb = (C.c_void_p * gB.ncontig)(*[x.ctypes.data + 1 for x in B])
    L = OrcLayout(*layout)
    P = OrcParams(chain_break, chain_min, align_min, align_rate)
    o.orc_new_result.restype = C.c_void_p
    R = C.c_void_p(o.orc_new_result())
    recs = np.ascontiguousarray(recs, dtype=np.uint64)
    p1 = np.ascontiguousarray(perm1, dtype=np.int32)
    p2 = np.ascontiguousarray(perm2, dtype=np.int32)
    n = o.orc_search(recs.ctypes.data_as(C.c_void_p), C.c_int64(len(recs)), C.byref(L), C.byref(P),
                     C.byref(spec), p1.ctypes.data_as(C.c_void_p), p2.ctypes.data_as(C.c_void_p),
                     pa, pac, gA.clen.ctypes.data_as(C.c_void_p), pb, gB.clen.ctypes.data_as(C.c_void_p), R)
    o.orc_result_ovls.restype = C.c_void_p
    o.orc_result_traces.restype = C.c_void_p
    o.orc_result_hits.restype = C.c_int64
    o.orc_result_ovls.argtypes = o.orc_result_traces.argtypes = o.orc_result_hits.argtypes = [C.c_void_p]
    nhit = o.orc_result_hits(R)
    if n > 0:
        ov = np.ctypeslib.as_array(C.cast(o.orc_result_ovls(R), C.POINTER(C.c_uint8)),
                                   shape=(n * OVL_DT.itemsize,)).view(OVL_DT).copy()
        tl = int((ov["toff"] + ov["tlen"]).max())
        tp = np.ctypeslib.as_array(C.cast(o.orc_result_traces(R), C.POINTER(C.c_uint8)), shape=(max(tl, 1),)).copy()
    else:
        ov = np.zeros(0, dtype=OVL_DT)
        tp = np.zeros(0, dtype=np.uint8)
    o.orc_free_result.argtypes = [C.c_void_p]
    o.orc_free_result(R)
    return ov, tp, nhit


def pack_overlaps(ov, tp, rank1, rank2, jb, ib):
    """oracle alignments (discovery order) -> the packed record buffer the device stage emits, so the
    product's host filter can be run on them"""
    from fastga_b200 import lib
    parts = []
    for i, r in enumerate(ov):
        pk = (int(r["comp"]) << (jb + ib)) | (int(rank1[r["aread"]]) << jb) | int(rank2[r["bread"]])
        h = np.array([i, 0, pk, r["abpos"], r["bbpos"], r["aepos"], r["bepos"], r["diffs"], r["tlen"], 0],
                     dtype=np.int32)
        tr = bytes(tp[int(r["toff"]):int(r["toff"]) + int(r["tlen"])])
        tr += b"\0" * ((-len(tr)) % 8)
        parts.append(h.tobytes())
        parts.append(tr)
    buf = np.frombuffer(b"".join(parts), dtype=np.uint8) if parts else np.zeros(0, np.uint8)
    return lib.overlaps_from_buffer(buf)


def seed_layout(gA, gB):
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    ab = int(amx + bmx).bit_length()
    return (ab, max(ab - 6, 1), int(max(gB.ncontig - 1, 1)).bit_length(),
            int(max(gA.ncontig - 1, 1)).bit_length(), amx, bmx)


def oracle_pipeline(gA, gB, **kw):
    """The whole path through the CPU oracle + the product's host filter.  Returns a dict."""
    from fastga_b200 import lib
    pa, ra = contig_rank(gA.clen)
    pb, rb = contig_rank(gB.clen)
    tA, sA = gix_build(gA, ra)
    tB, sB = gix_build(gB, rb)
    seeds, sumlen = merge(tA, tB, sB, kw.get("freq", 10))
    layout = seed_layout(gA, gB)
    recs = seed_records(seeds, layout)
    skw = {k: v for k, v in kw.items() if k in ("chain_break", "chain_min", "align_min", "align_rate")}
    ov, tp, nhit = search(recs, layout, gA, gB, pa, pb, gA.freq, **skw)
    O = pack_overlaps(ov, tp, ra, rb, layout[2], layout[3])
    al = lib.filter_overlaps(O.h, pa, pb, layout[2], layout[3])
    return dict(tabA=tA, tabB=tB, pstartA=sA, pstartB=sB, nseeds=len(seeds), sumlen=sumlen, seedrecs=recs,
                nhit=nhit, nraw=len(ov), alns=al, lines=al.canonical_lines(), perm1=pa, perm2=pb)


def oracle_pipeline_self(g, **kw):
    """SELF mode (FastGA A) through the CPU oracle + the product's host filter (groundwork for
    SURVEY row a-7; no CUDA path uses it yet)."""
    from fastga_b200 import lib
    pa, ra = contig_rank(g.clen)
    t, s = gix_build(g, ra)
    seeds, sumlen = self_merge(t, s, kw.get("freq", 10))
    layout = seed_layout(g, g)
    recs = seed_records(seeds, layout)
    o = orc()
    o.orc_set_self(1)
    try:
        ov, tp, nhit = search(recs, layout, g, g, pa, pa, g.freq)
    finally:
        o.orc_set_self(0)
    O = pack_overlaps(ov, tp, ra, ra, layout[2], layout[3])
    al = lib.filter_overlaps(O.h, pa, pa, layout[2], layout[3])
    return dict(nseeds=len(seeds), sumlen=sumlen, nhit=nhit, nraw=len(ov), alns=al, lines=al.canonical_lines())
